"""Forward plan of the SAVSR hot path on libsavsr_sm100 (host side, Python like the reference).

A ``Plan`` is built once per (batch, h, w, scale, weights-version).  It packs the weights into the
tensor-core layouts, lays the activations out in bf16 NHWC arenas, pre-computes the SATU index vectors
and per-scale MLP table, and records the ordered list of C-ABI kernel launches that make up
``SAVSR.forward`` (reference: lbasicsr/archs/savsr_arch.py:692-742).  ``run()`` replays that list on the
current CUDA stream; ``run_graph()`` replays a CUDA graph captured from it.

The two propagation directions (f2p / p2f, savsr_arch.py:708-719) are independent chains, so every
launch of the propagation phase batches both directions (and the 3 or 5 per-frame streams of a
ResidualBlock) as "groups" of one grouped implicit-GEMM launch instead of using two streams.

PyTorch is used here only for device memory and streams.  There is no CPU path.
"""
from __future__ import annotations

import os

import ctypes as C
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _capi as K, colour

BN_EPS = 1e-5
IO_MODES = ("f32", "bgr_u8", "bgr_u8_frames", "bgr48_frames")
FRAME_MODES = {"bgr_u8_frames": torch.uint8, "bgr48_frames": torch.uint16}     # I/O modes that read frames in place, and their sample type


def normalize_scale(scale) -> Tuple[float, float]:
    if isinstance(scale, (int, float)):
        return (scale, scale)
    s = tuple(scale)
    if len(s) != 2:
        raise ValueError(f"scale must be a number or a (s_h, s_w) pair, got {scale!r}")
    return (s[0], s[1])


def get_hw(h: int, w: int, scale) -> Tuple[int, int]:
    """savsr_arch.py:745-751: python round() (half-to-even) on the python float product."""
    s = normalize_scale(scale)
    return round(h * s[0]), round(w * s[1])


_contexts: Dict[int, K.Context] = {}


def context(device_index: int) -> K.Context:
    """One savsr_ctx per device.  Bring-up knobs come from the environment HERE (the library itself reads none)."""
    if device_index not in _contexts:
        c = K.Context(device_index)
        if os.environ.get("SAVSR_BIGK_ALL") is not None:
            c.set_option(K.OPT_BIGK_ALL, int(os.environ["SAVSR_BIGK_ALL"] != "0"))
        if os.environ.get("SAVSR_BIGK_ISSUERS") is not None:
            c.set_option(K.OPT_BIGK_ISSUERS, int(os.environ["SAVSR_BIGK_ISSUERS"]))
        if os.environ.get("SAVSR_PDL") is not None:
            c.set_option(K.OPT_PDL, int(os.environ["SAVSR_PDL"] != "0"))
        _contexts[device_index] = c
    return _contexts[device_index]


class pdl:
    """`with pdl(ctx, on)`: launches issued (or captured) inside use programmatic dependent launch (SAVSR_OPT_PDL): the next kernel's CTAs are
    scheduled while the current one drains.  Worth 1-2 % on chains of microsecond-sized launches (the training step at 4 x 64 x 64, b = 1
    inference), nothing on long launches.  SAVSR_PDL=0 / 1 in the environment overrides the choice."""

    def __init__(self, ctx: K.Context, on: bool):
        self.ctx = ctx
        env = os.environ.get("SAVSR_PDL")
        self.on = int(on if env is None else env != "0")

    def __enter__(self):
        self.prev = self.ctx.lib.savsr_ctx_get_option(self.ctx.handle, K.OPT_PDL)
        self.ctx.set_option(K.OPT_PDL, self.on)
        return self

    def __exit__(self, *exc):
        self.ctx.set_option(K.OPT_PDL, max(self.prev, 0))
        return False


class WeightStore:
    """Everything a plan derives from the weights alone -- packed tensor-core layouts, folded BatchNorm, zero-expanded
    first-layer filters -- keyed by name and shared by all plans of one (module, device, precision, weights version).
    A new (batch, h, w, scale) plan then only allocates its arenas and records its launch list (the reference YAMLs sweep
    42-48 scales per run)."""

    def __init__(self, version: tuple = ()):
        self.version = version
        self.cache: Dict[tuple, torch.Tensor] = {}

    def get(self, key: tuple, make: Callable[[], torch.Tensor]) -> torch.Tensor:
        t = self.cache.get(key)
        if t is None:
            t = self.cache[key] = make()
        return t


class _Slots:
    """Arena slot allocator with reuse (program order == stream order, single stream)."""

    def __init__(self):
        self.free: List[int] = []
        self.n = 0

    def get(self) -> int:
        if self.free:
            return self.free.pop()
        self.n += 1
        return self.n - 1

    def get_many(self, k: int) -> List[int]:
        return [self.get() for _ in range(k)]

    def get_contiguous(self, k: int) -> int:
        s = self.n
        self.n += k
        return s

    def put(self, *slots: int) -> None:
        self.free.extend(slots)


def satu_hr_compose(P: Dict[str, torch.Tensor], device: torch.device):
    """Host-side composition of the linear chain fusion (1x1, 128->64) -> tail (3x3, 64->3), savsr_arch.py:374, 738, for
    savsr_satu_hr: rows k = (dy*3+dx)*3 + c.  Returns fp32 (Wc [32,64], Wcf [27,64], Wcs [27,64], Wv [27,32], zb [32]):
        Z[q][k] = S[q] Wcs^T + F[q] Wcf^T + V[q] Wv^T + zb ;   sr[p][c] = bt[c] + sum_tap Z[p + d_tap][tap*3+c]
    (computed in float64, rounded once)."""
    g = lambda name: P[name].detach().to(device, torch.float64)   # noqa: E731
    u = "upsample"
    Wf = g(u + ".fusion.weight").view(64, 128)
    bf = g(u + ".fusion.bias")
    Wt = g("tail.weight").permute(2, 3, 0, 1).reshape(27, 64)                           # [(dy,dx,c)][o]
    comb = Wt @ Wf                                                                        # [27, 128]: in = [sta_s | fea] (374: sta first)
    Wcs, Wcf = comb[:, :64], comb[:, 64:]
    We = g(u + ".weight_expand").view(4, 64, 8).permute(1, 0, 2).reshape(64, 32)         # [c][e*8+k]
    Wv = Wcf @ We                                                                         # fea = V We^T + F
    Wc = g(u + ".weight_compress").reshape(32, 64)                                       # rows e*8+k
    zb = torch.zeros(32, dtype=torch.float64, device=device)
    zb[:27] = Wt @ bf
    return Wc.float(), Wcf.float().contiguous(), Wcs.float().contiguous(), Wv.float(), zb.float()


def satu_hr_pack(parts, fmt: int, device: torch.device) -> torch.Tensor:
    """The four B operands of savsr_satu_hr (Wc | Wcf | Wcs | Wv) as [32 rows][128 B] K-major 128-byte-swizzled 16-bit tiles
    (16 KB): the 16-byte chunk c of row n sits at chunk position c ^ (n & 7)."""
    dt = torch.float16 if fmt == K.FMT_FP16 else torch.bfloat16
    n = torch.arange(32, device=device).view(32, 1)
    pos = torch.arange(8, device=device).view(1, 8) ^ (n & 7)                            # [32, 8]
    tiles = []
    for m in parts[:4]:
        full = torch.zeros(32, 64, device=device)
        full[:m.shape[0], :m.shape[1]] = m
        src = full.to(dt).view(32, 8, 8)
        tile = torch.zeros_like(src)
        tile.scatter_(1, pos.view(32, 8, 1).expand(32, 8, 8), src)
        tiles.append(tile.reshape(-1))
    return torch.cat(tiles).view(torch.uint8).contiguous()


class Plan:
    """I/O modes (`io`): "f32" stages the module's forward contract, x fp32 [B,7,3,h,w] RGB in [0, 1] -> out fp32 [B,3,H,W];
    "bgr_u8" stages decoded 8-bit video, x uint8 [B,7,h,w,3] BGR -> out uint8 [B,H,W,3] BGR, the image tensor2img makes of the
    fp32 output of x / 255; "bgr_u8_frames" has no input staging: it reads B*7 uint8 BGR [h,w,3] frames in place through a device
    table of frame pointers (`frame_table`, written per forward by forward_frames_into) -> out uint8 [B,H,W,3] as "bgr_u8";
    "bgr48_frames" is the same for deep video: B*7 uint16 bgr48 [h,w,3] frames, each value v entering as v / 65535 -> out uint16
    [B,H,W,3], the fp32 output clamped, * 65535 and rounded half to even.
    The modes differ only in their first and last launch (savsr_pack_frames[_u8[_table] | _u16_table], savsr_satu_hr[...])."""
    io = "f32"

    def __init__(self, params: Dict[str, torch.Tensor], batch: int, h: int, w: int, scale, device: torch.device,
                 conv_impl: str = "tap", num_frame: int = 7, taps: Optional[Sequence[str]] = None, precision: str = "bf16",
                 store: Optional[WeightStore] = None, io: str = "f32"):
        if device.type != "cuda":
            raise K.SavsrError("savsr_b200 runs on CUDA (sm_100a) only; there is no CPU fallback")
        if num_frame != 7:
            raise NotImplementedError("only the shipped 7-frame configuration is implemented")
        if h < 2 or w < 2:
            raise ValueError(f"LR frames must be at least 2x2, got {h}x{w}")
        if io not in IO_MODES:
            raise ValueError(f"io must be one of {IO_MODES}, got {io!r}")
        self.device = device
        self.ctx = context(device.index if device.index is not None else torch.cuda.current_device())
        self.lib = self.ctx.lib
        self.impl = K.IMPL_NAMES[conv_impl]
        if precision not in K.FMT_NAMES:
            raise ValueError(f"precision must be one of {sorted(K.FMT_NAMES)}, got {precision!r}")
        self.fmt = K.FMT_NAMES[precision]
        self.io = io
        self.B, self.h, self.w, self.t = batch, h, w, num_frame
        self.scale = normalize_scale(scale)
        self.hp, self.wp = h + (h & 1), w + (w & 1)
        self.H, self.W = get_hw(h, w, self.scale)
        self.P = params
        self._keep: List[object] = []   # tensors / ctypes arrays referenced by raw pointers
        self._pack_src: List[torch.Tensor] = []
        self.ops: List[Callable[[int], int]] = []
        self.op_meta: List[Tuple[str, float, int, str]] = []   # (kind, algorithmic FLOPs, kernel launches, detail) per op
        self.n_launches = 0
        self.taps = set(taps or ())
        self.tap_bufs: Dict[str, torch.Tensor] = {}
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.store = store if store is not None else WeightStore()
        self.nbytes = 0                          # device memory owned by this plan (arenas, scratch, I/O staging)
        self._pool_cache: Dict[str, int] = {}
        self._osa_cache: Dict[str, Tuple[K.OsaParams, int, int]] = {}
        self.cplan: Optional[K.CPlan] = K.CPlan(self.ctx) if hasattr(K, "CPlan") and hasattr(self.lib, "savsr_plan_create") else None
        self._recorded = 0
        with torch.cuda.device(device), torch.no_grad():
            self.ctx.set_format(self.fmt)
            self._build()
            if self.cplan is not None:
                if self._recorded == len(self.ops):
                    out_bytes = self.out.numel() * self.out.element_size()
                    if self.io in FRAME_MODES:
                        set_io = self.lib.savsr_plan_set_io_u8_table if self.io == "bgr_u8_frames" else self.lib.savsr_plan_set_io_u16_table
                        K.check(set_io(self.cplan.handle, self.frame_table.data_ptr(), self.frame_table.numel(), self.out.data_ptr(), out_bytes,
                                       self.fmt))
                    else:
                        set_io = self.lib.savsr_plan_set_io_u8 if self.io == "bgr_u8" else self.lib.savsr_plan_set_io
                        K.check(set_io(self.cplan.handle, self.x_in.data_ptr(), self.x_in.numel() * self.x_in.element_size(), self.out.data_ptr(),
                                       out_bytes, self.fmt))
                else:
                    self.cplan = None                       # an op without a C-side record: keep the Python loop

    # ------------------------------------------------------------------ memory helpers
    def _buf(self, *shape, dtype=torch.float32) -> torch.Tensor:
        t = torch.empty(*shape, dtype=dtype, device=self.device)
        self._keep.append(t)
        self.nbytes += t.numel() * t.element_size()
        return t

    def _p(self, name: str) -> torch.Tensor:
        t = self.P[name]
        if t.device != self.device or t.dtype != torch.float32 or not t.is_contiguous():
            t = t.detach().to(self.device, torch.float32).contiguous()
        self._keep.append(t)
        return t

    def _ptr(self, name: str) -> int:
        return self._p(name).data_ptr()

    def _derived(self, key, make: Callable[[], torch.Tensor]) -> torch.Tensor:
        """fp32 device tensor computed from the weights alone (folded BN, zero-expanded filters ...), shared through the store."""
        return self.store.get(("derived", key), lambda: make().detach().to(self.device, torch.float32).contiguous())

    def _dev(self, key, make: Callable[[], torch.Tensor]) -> int:
        return self._derived(key, make).data_ptr()

    def _packp(self, name: str) -> int:
        """Packed copy of the conv parameter `name` (shared: the five propagation iterations and every plan use one copy)."""
        return self._pack(name, lambda: self._p(name))

    def _pack(self, key, make: Callable[[], torch.Tensor], n_tile: int = 64, co_pad: Optional[int] = None,
              rows: int = K.ROWS_QUAD) -> int:
        """fp32 OIHW -> packed 16-bit tensor-core layout; returns the device pointer.  `rows`: row order of n_tile 64
        blocks -- QUAD for everything savsr_conv consumes, LINEAR for the SATU expert GEMMs.  Cached in the store by `key`."""
        def build() -> torch.Tensor:
            w = make().detach().to(self.device, torch.float32).contiguous()
            co_real, ci, ks, _ = w.shape
            co = co_pad or co_real
            out = torch.empty(self.lib.savsr_packed_weight_bytes(co, ci, ks), dtype=torch.uint8, device=self.device)
            K.check(self.lib.savsr_pack_conv_weight(w.data_ptr(), co_real, co, ci, ks, n_tile, self.fmt, rows, out.data_ptr(),
                                                    torch.cuda.current_stream(self.device).cuda_stream))
            self._pack_src.append(w)                 # the source must outlive the asynchronous pack kernel
            return out
        return self.store.get(("packed", key, n_tile, co_pad, rows, self.fmt), build).data_ptr()

    # ------------------------------------------------------------------ op emitters
    def _emit(self, fn: Callable[[int], int], launches: int = 1, kind: str = "other", flops: float = 0.0,
              detail: str = "", rec: Optional[Callable[[object], int]] = None) -> None:
        """Append one op to the launch list.  `rec` records the same launch into the C-side plan (savsr_plan), which replays the whole
        list with one call (savsr_plan_run / savsr_forward); the Python closures stay for per-op timing and debugging."""
        self.ops.append(fn)
        self.op_meta.append((kind, flops, launches, detail))
        self.n_launches += launches
        if rec is not None and self.cplan is not None:
            K.check(rec(self.cplan.handle))
            self._recorded += 1

    def _group(self, src: Sequence[int], dst: int, weight: int, bias: int = 0, act: int = K.ACT_NONE, slope: float = 0.2,
               res1: int = -1, res2: int = -1, res2_scale: float = 0.0, wstride: int = 0, mask: int = 0, pool: int = 0,
               aux: int = 0, src_channels: int = 0) -> K.ConvGroup:
        g = K.ConvGroup()
        for i, s in enumerate(src):
            g.src_slot[i] = s
        g.nsrc = len(src)
        g.dst_slot, g.res1_slot, g.res2_slot, g.res2_scale = dst, res1, res2, res2_scale
        g.act, g.slope = act, slope
        g.weight, g.weight_sample_stride = weight, wstride
        g.bias, g.mask, g.pool, g.aux_dst = bias or None, mask or None, pool or None, aux or None
        g.src_channels = src_channels
        return g

    def _conv(self, arena: K.Arena, groups: Sequence[K.ConvGroup], ksize: int = 3, n_tile: int = 64,
              dst_mode: int = K.DST_ARENA, alg_ci: Optional[Sequence[int]] = None, alg_co: Optional[int] = None,
              kind: Optional[str] = None) -> None:
        """Emit one batched savsr_conv launch.  `alg_ci` / `alg_co`: ALGORITHMIC input channels per group / output channels,
        where they differ from the padded GEMM shape (first layer: 3 and 6 of 64) -- the FLOP count of the
        roofline uses the reference's channel counts (SURVEY.md 8d), never the zero padding."""
        arr = (K.ConvGroup * len(groups))(*groups)
        self._keep.append(arr)
        lib, ctx, ah, n, impl = self.lib, self.ctx.handle, arena.handle, len(groups), self.impl
        co = alg_co if alg_co is not None else (64 if n_tile == 64 else 16)      # real output channels
        ci = list(alg_ci) if alg_ci is not None else [64 * g.nsrc for g in groups]
        flops = 2.0 * self.B * arena.height * arena.width * co * ksize * ksize * sum(ci)
        osa = any(g.weight_sample_stride != 0 for g in groups)
        self._emit(lambda st: lib.savsr_conv(ctx, ah, arr, n, ksize, n_tile, dst_mode, impl, st),
                   kind=kind or f"conv{ksize}x{ksize}_n{n_tile}", flops=flops,
                   detail=f"g{n}s{groups[0].nsrc}" + ("osa" if osa else ""),
                   rec=lambda cp: lib.savsr_plan_add_conv(cp, ah, arr, n, ksize, n_tile, dst_mode, impl))

    def _tap(self, name: str, arena: str, slot: int) -> None:
        """Test/debug hook: if `name` was requested in `taps`, snapshot the slot (fp32 NCHW) right here in the
        program, before later stages recycle it.  Not emitted in production plans."""
        if name not in self.taps:
            return
        a = self.lr
        buf = self._buf(self.B, 64, a.height, a.width)
        self.tap_bufs[name] = buf
        lib, ah, ptr = self.lib, a.handle, buf.data_ptr()
        self._emit(lambda st: lib.savsr_arena_export(ah, slot, ptr, st), kind="debug_tap", rec=lambda cp: lib.savsr_plan_add_arena_export(cp, ah, slot, ptr))

    def _osa_params(self, prefix: str, nsrc: int, pools: Sequence[int]) -> Tuple[K.OsaParams, int, int]:
        if prefix in self._osa_cache:
            return self._osa_cache[prefix]
        ci, co = 64 * nsrc, 64
        att = max(int(ci * 0.0625), 16)
        a = prefix + ".attention"
        def bn_s():
            return self._p(a + ".bn.weight") / torch.sqrt(self._p(a + ".bn.running_var") + BN_EPS)

        def bn_b():
            return self._p(a + ".bn.bias") - self._p(a + ".bn.running_mean") * bn_s()
        o = K.OsaParams()
        o.ci, o.co, o.att = ci, co, att
        o.bank = self._ptr(prefix + ".weight")
        o.r0_w, o.r0_b = self._ptr(prefix + ".scale_routing.0.weight"), self._ptr(prefix + ".scale_routing.0.bias")
        o.r2_w, o.r2_b = self._ptr(prefix + ".scale_routing.2.weight"), self._ptr(prefix + ".scale_routing.2.bias")
        o.fc_w = self._ptr(a + ".fc.weight")
        o.bn_scale, o.bn_shift = self._dev(a + ".bn_scale", bn_s), self._dev(a + ".bn_shift", bn_b)
        o.ch_w, o.ch_b = self._ptr(a + ".channel_fc.weight"), self._ptr(a + ".channel_fc.bias")
        o.fl_w, o.fl_b = self._ptr(a + ".filter_fc.weight"), self._ptr(a + ".filter_fc.bias")
        o.sp_w, o.sp_b = self._ptr(a + ".spatial_fc.weight"), self._ptr(a + ".spatial_fc.bias")
        o.kn_w, o.kn_b = self._ptr(a + ".kernel_fc.weight"), self._ptr(a + ".kernel_fc.bias")
        for i, pp in enumerate(pools):
            o.pool[i] = pp
        scratch = self._buf(self.B, 5 * ci + 192)
        packed = self._buf(self.B, co * ci * 9 * 2, dtype=torch.uint8)
        o.scratch, o.packed = scratch.data_ptr(), packed.data_ptr()
        self.osa_scratch[prefix] = scratch
        self._osa_cache[prefix] = (o, packed.data_ptr(), co * ci * 9 * 2)
        return self._osa_cache[prefix]

    def _osa_prologue(self, convs: Sequence[K.OsaParams]) -> None:
        arr = (K.OsaParams * len(convs))(*convs)
        self._keep.append(arr)
        inv_h = float(np.float32(1.0) / np.float32(self.scale[0]))
        inv_w = float(np.float32(1.0) / np.float32(self.scale[1]))
        lib, ctx, n, B = self.lib, self.ctx.handle, len(convs), self.B
        npart, npix = self.lr.tiles * 4, self.hp * self.wp
        self._emit(lambda st: lib.savsr_osa_prologue(ctx, arr, n, B, npart, npix, inv_h, inv_w, st), launches=4, kind="osa_prologue",
                   rec=lambda cp: lib.savsr_plan_add_osa_prologue(cp, arr, n, B, npart, npix, inv_h, inv_w))

    def _pool(self, key: str) -> int:
        """Partial-sum buffer [B][tiles*4][64] written by a conv epilogue (cached per producing conv)."""
        if key not in self._pool_cache:
            self._pool_cache[key] = self._buf(self.B, self.lr.tiles * 4, 64).data_ptr()
        return self._pool_cache[key]

    # ------------------------------------------------------------------ program construction
    def _residual_block(self, prefixes: Sequence[str], xs: Sequence[Sequence[int]], outs: Sequence[Sequence[int]],
                        tmp: Sequence[Sequence[int]], base: Sequence[int]) -> None:
        """ResidualBlock.forward (savsr_arch.py:399-415) for len(prefixes) independent blocks at once.
        xs[d][i] -> outs[d][i]; tmp[d][i] holds x1, base[d] the merged feature."""
        lr = self.lr
        nfr = len(xs[0])
        use_os = (prefixes[0] + ".osconv.weight") in self.P
        L = K.ACT_LRELU
        pools = [[self._pool(f"{p}.conv0.{i}") if use_os else 0 for i in range(nfr)] for p in prefixes]
        self._conv(lr, [self._group([xs[d][i]], tmp[d][i], self._packp(f"{p}.conv0.{i}.weight"),
                                    self._ptr(f"{p}.conv0.{i}.bias"), act=L, pool=pools[d][i])
                        for d, p in enumerate(prefixes) for i in range(nfr)])
        if use_os:
            osa = [self._osa_params(p + ".osconv", nfr, pools[d]) for d, p in enumerate(prefixes)]
            self._osa_prologue([o[0] for o in osa])
            self._conv(lr, [self._group(tmp[d], base[d], osa[d][1], act=L, wstride=osa[d][2]) for d in range(len(prefixes))])
        else:
            self._conv(lr, [self._group(tmp[d], base[d], self._packp(p + ".conv1.weight"), self._ptr(p + ".conv1.bias"), act=L)
                            for d, p in enumerate(prefixes)], ksize=1)
        self._conv(lr, [self._group([base[d], tmp[d][i]], outs[d][i], self._packp(f"{p}.conv2.{i}.weight"),
                                    self._ptr(f"{p}.conv2.{i}.bias"), act=L, res1=xs[d][i])
                        for d, p in enumerate(prefixes) for i in range(nfr)])

    def _build(self) -> None:
        P, B, t = self.P, self.B, self.t
        lib, ctx = self.lib, self.ctx.handle
        L = K.ACT_LRELU
        self.osa_scratch: Dict[str, torch.Tensor] = {}
        nf = 64
        # ---- arenas: slot count is discovered by a dry layout pass (slot ids only), then allocated.
        sl = _Slots()
        zero = sl.get()
        FR = sl.get()                                              # the 7 LR frames as one 21(+43 zero)-channel slot
        dirs = ("f2p_win", "p2f_win")
        n_it = t - 3 + 1
        F = [[sl.get() for _ in range(n_it)] for _ in dirs]        # unit outputs, kept for the l2 fusion
        S0 = [sl.get_many(2) for _ in dirs]
        S1 = [sl.get_many(3) for _ in dirs]
        S2 = [sl.get_many(3) for _ in dirs]
        T = [sl.get_many(3) for _ in dirs]
        Bs = [sl.get() for _ in dirs]
        # l2 / reconstruction reuse the propagation scratch slots
        pool_free = [s for d in range(2) for s in (S0[d] + S1[d] + S2[d] + T[d])] + Bs
        extra_needed = 5 + 5 + 5 + 1 + 2 + 1 + 6 + 2
        while len(pool_free) < extra_needed:
            pool_free.append(sl.get())
        self.n_lr_slots = sl.n
        self.arena_lr_t = self._buf(self.n_lr_slots * B, self.hp, self.wp, 64, dtype=torch.bfloat16)
        self.arena_lr_t.zero_()                  # the zero slot must be zero; the rest so that activation_absmax never reads stale memory
        self.lr = K.Arena(self.ctx, self.arena_lr_t.data_ptr(), self.n_lr_slots, B, self.hp, self.wp)
        lr = self.lr
        if self.io in FRAME_MODES:
            self.x_in = None
            self.frame_table = self._buf(B * t, dtype=torch.int64)         # const uint8_t* / uint16_t* [B][t], rewritten before every forward
            self.out = self._buf(B, self.H, self.W, 3, dtype=FRAME_MODES[self.io])
            xin = self.frame_table.data_ptr()
        else:
            if self.io == "bgr_u8":
                self.x_in = self._buf(B, t, self.h, self.w, 3, dtype=torch.uint8)
                self.out = self._buf(B, self.H, self.W, 3, dtype=torch.uint8)
            else:
                self.x_in = self._buf(B, t, 3, self.h, self.w)
                self.out = self._buf(B, 3, self.H, self.W)
            xin = self.x_in.data_ptr()
        sfx = {"f32": "", "bgr_u8": "_u8", "bgr_u8_frames": "_u8_table", "bgr48_frames": "_u16_table"}[self.io]   # the first and the last launch; everything between is shared
        pack_frames, add_pack_frames = getattr(lib, "savsr_pack_frames" + sfx), getattr(lib, "savsr_plan_add_pack_frames" + sfx)
        satu_hr, add_satu_hr = getattr(lib, "savsr_satu_hr" + sfx), getattr(lib, "savsr_plan_add_satu_hr" + sfx)

        # ---- 1. bi-directional propagation (savsr_arch.py:703-719), both directions per launch
        lrh0, hh0, ww0 = lr.handle, self.h, self.w
        self._emit(lambda st: pack_frames(ctx, lrh0, xin, t, hh0, ww0, FR, st), kind="pack_frames",
                   rec=lambda cp: add_pack_frames(cp, lrh0, xin, t, hh0, ww0, FR))
        hpast = [zero, zero]
        for idx in range(n_it):
            centre = [t - 1 - 1 - idx, idx + 1]                     # f2p walks back, p2f forward
            # first-layer convs on the tensor-core kernel: the packed-frames slot is the single source and the
            # 3/6-channel filters are zero-expanded to the frame channels they read (savsr_arch.py:447-457)
            fgroups = []
            for d, p in enumerate(dirs):
                c = centre[d]

                def wc(p=p, c=c):
                    wz = torch.zeros(64, 64, 3, 3, device=self.device)
                    wz[:, 3 * c:3 * c + 3] = self._p(p + ".conv_c.weight")
                    return wz

                def ws(p=p, c=c):
                    wz = torch.zeros(64, 64, 3, 3, device=self.device)
                    wsup = self._p(p + ".conv_sup.weight")
                    wz[:, 3 * (c - 1):3 * (c - 1) + 3] = wsup[:, 0:3]
                    wz[:, 3 * (c + 1):3 * (c + 1) + 3] = wsup[:, 3:6]
                    return wz
                # the frames slot carries 7 x 3 = 21 channels: the K loop runs over the first 32 only
                fgroups.append(self._group([FR], S0[d][0], self._pack((p, "conv_c@", c), wc), self._ptr(p + ".conv_c.bias"), act=L, src_channels=32))
                fgroups.append(self._group([FR], S0[d][1], self._pack((p, "conv_sup@", c), ws), self._ptr(p + ".conv_sup.bias"), act=L, src_channels=32))
            # algorithmic input channels of these launches are 3 and 6, not the 64 of the zero-expanded filters
            self._conv(lr, fgroups, alg_ci=[3, 6, 3, 6])
            cur = [[S0[d][0], S0[d][1], hpast[d]] for d in range(2)]
            sets = [S1, S2]
            for j in range(4):
                nxt = sets[j % 2]
                self._residual_block([f"{p}.blocks.{j}" for p in dirs], cur, nxt, T, Bs)
                cur = [list(nxt[d]) for d in range(2)]
            self._conv(lr, [self._group(cur[d], F[d][idx], self._packp(p + ".merge.weight"), self._ptr(p + ".merge.bias"))
                            for d, p in enumerate(dirs)])
            hpast = [F[0][idx], F[1][idx]]
        self._tap("f2p_last", "lr", F[0][n_it - 1])
        self._tap("p2f_last", "lr", F[1][n_it - 1])

        # ---- 2. pyramid fusion, WindowUnit_l2 (savsr_arch.py:485-501, 721-723)
        free = list(pool_free)
        take = lambda k: [free.pop() for _ in range(k)]
        Gx, Gy, T5 = take(5), take(5), take(5)
        B5, = take(1)
        M = take(2)
        A, = take(1)
        p2 = "h_win.0"
        # h_f2p_list.insert(0, .) reverses the f2p order: list position i <- unit idx = n_it-1-i
        self._conv(lr, [self._group([F[0][n_it - 1 - i], F[1][i]], Gx[i], self._packp(f"{p2}.conv_h.{i}.weight"),
                                    self._ptr(f"{p2}.conv_h.{i}.bias"), act=L) for i in range(5)])
        cur5, nxt5 = Gx, Gy
        for j in range(2):
            self._residual_block([f"{p2}.blocks.{j}"], [cur5], [nxt5], [T5], [B5])
            cur5, nxt5 = nxt5, cur5
        wm = self._packp(p2 + ".merge.weight")
        half = 5 * 9 * 8192
        bm = self._p(p2 + ".merge.bias")
        self._conv(lr, [self._group(cur5, M[k], wm + k * half, bm[64 * k:].data_ptr()) for k in range(2)])
        self._tap("h_win0", "lr", M[0]); self._tap("h_win1", "lr", M[1])
        self._conv(lr, [self._group(M, A, self._packp("h_win_conv_h.weight"), self._ptr("h_win_conv_h.bias"), act=L)])
        self._tap("align", "lr", A)
        free += Gx + Gy + T5 + [B5] + M

        # ---- 3. reconstruction: 4 x (ResidualGroup -> OSAdapt -> + gamma * share) (savsr_arch.py:727-734)
        gamma = float(self._p("gamma").item())
        X0, X1, T1, T2, R, Hs = take(6)
        in16 = self._buf(B, self.hp * self.wp, 16)
        half0 = self._buf(B, (self.hp // 2) * (self.wp // 2), 16)
        half1 = self._buf(B, (self.hp // 2) * (self.wp // 2), 16)
        maskb = self._buf(B, self.hp * self.wp)
        ca_y = self._buf(B, 64).data_ptr()
        npart = lr.tiles * 4
        lrh = lr.handle
        h_cur = A                                   # share_source / align_feat stay in slot A to the end
        for gi in range(4):
            x, xa, xb = h_cur, X0, X1               # RCAB chain ping-pongs X0/X1, h_cur is kept for the group residual
            for r in range(8):
                pr = f"RG.{gi}.residual_group.{r}.rcab"
                self._conv(lr, [self._group([x], T1, self._packp(pr + ".0.weight"), self._ptr(pr + ".0.bias"), act=K.ACT_RELU)])
                pl = self._pool(pr + ".2")
                self._conv(lr, [self._group([T1], T2, self._packp(pr + ".2.weight"), self._ptr(pr + ".2.bias"), pool=pl)])
                w1, b1 = self._ptr(pr + ".3.attention.1.weight"), self._ptr(pr + ".3.attention.1.bias")
                w2, b2 = self._ptr(pr + ".3.attention.3.weight"), self._ptr(pr + ".3.attention.3.bias")
                self._emit(lambda st, x=x, xa=xa, pl=pl, w1=w1, b1=b1, w2=w2, b2=b2:
                           lib.savsr_ca_scale_residual(ctx, lrh, T2, x, xa, pl, npart, w1, b1, w2, b2, ca_y, st),
                           launches=2, kind="ca_scale_residual",
                           rec=lambda cp, x=x, xa=xa, pl=pl, w1=w1, b1=b1, w2=w2, b2=b2:
                           lib.savsr_plan_add_ca_scale_residual(cp, lrh, T2, x, xa, pl, npart, w1, b1, w2, b2, ca_y))
                x, xa, xb = xa, xb, xa
            plr = self._pool(f"RG.{gi}.conv")
            self._conv(lr, [self._group([x], R, self._packp(f"RG.{gi}.conv.weight"), self._ptr(f"RG.{gi}.conv.bias"),
                                        res1=h_cur, pool=plr)])
            self._tap(f"rg{gi}", "lr", R)
            # OSAdapt (savsr_arch.py:186-214): mask branch, adapted = OSA-Conv(x); h = x + adapted * mask + gamma * share
            pa = f"adapt.{gi}"
            m = pa + ".mask"

            def fold(conv: str, bn: str):
                """conv + eval-mode BatchNorm -> (lazy folded weight, lazy folded bias), cached in the weight store"""
                def sc():
                    return self._p(bn + ".weight") / torch.sqrt(self._p(bn + ".running_var") + BN_EPS)
                return (lambda: self._p(conv + ".weight") * sc().view(-1, 1, 1, 1),
                        lambda: (self._p(conv + ".bias") - self._p(bn + ".running_mean")) * sc() + self._p(bn + ".bias"))
            w0, b0 = fold(m + ".0", m + ".1")
            wa, ba = fold(m + ".4", m + ".5")
            wb, bb = fold(m + ".7", m + ".8")
            wc, bc = fold(m + ".11", m + ".12")
            self._conv(lr, [self._group([R], 0, self._pack(m + ".0+bn", w0, n_tile=16), self._dev(m + ".0+bn.bias", b0), act=K.ACT_RELU,
                                        aux=in16.data_ptr())], n_tile=16, dst_mode=K.DST_AUX16)
            args = (ctx, in16.data_ptr(), B, self.hp, self.wp, self._dev(m + ".4+bn.w", wa), self._dev(m + ".4+bn.b", ba),
                    self._dev(m + ".7+bn.w", wb), self._dev(m + ".7+bn.b", bb), self._dev(m + ".11+bn.w", wc), self._dev(m + ".11+bn.b", bc),
                    half0.data_ptr(), half1.data_ptr(), maskb.data_ptr())
            self._emit(lambda st, args=args: lib.savsr_osadapt_mask(*args, st), launches=3, kind="osadapt_mask",
                       rec=lambda cp, args=args: lib.savsr_plan_add_osadapt_mask(cp, *args[1:]))
            osa = self._osa_params(pa + ".adapt", 1, [plr])
            self._osa_prologue([osa[0]])
            self._conv(lr, [self._group([R], Hs, osa[1], wstride=osa[2], mask=maskb.data_ptr(), res1=R, res2=A, res2_scale=gamma)])
            self._tap(f"adapt{gi}", "lr", Hs)
            h_cur = Hs
        TR, = take(1)
        self._conv(lr, [self._group([h_cur], TR, self._packp("conv_last.weight"), self._ptr("conv_last.bias"), res1=A)])
        self._tap("trunk", "lr", TR)

        # ---- 4. SATU (savsr_arch.py:315-376) + tail + bilinear skip (738-739)
        u = "upsample"
        wkp = self._pack(u + ".kernel_conv.tapmajor",
                         lambda: self._p(u + ".kernel_conv.0.weight").view(64, 25, 64).permute(1, 0, 2).reshape(1600, 64, 1, 1))
        bkp = self._dev(u + ".kernel_conv.tapmajor.bias", lambda: self._p(u + ".kernel_conv.0.bias").view(64, 25).t().contiguous())
        STA, = take(1)
        lrh, hh, ww = lr.handle, self.h, self.w
        # kernel_conv + sta_conv in one kernel: the 25 per-pixel kernels stay in TMEM (savsr_arch.py:297-313, 326)
        kflops = 2.0 * B * self.hp * self.wp * 64 * 1600
        self._emit(lambda st: lib.savsr_satu_kconv_sta(ctx, lrh, A, TR, STA, hh, ww, wkp, bkp, 0.1, st), kind="satu_kconv_sta",
                   flops=kflops, rec=lambda cp: lib.savsr_plan_add_satu_kconv_sta(cp, lrh, A, TR, STA, hh, ww, wkp, bkp, 0.1))
        self._tap("satu_sta", "lr", STA)
        sw = K.SatuWeights()
        sw.body0_w, sw.body0_b = self._ptr(u + ".body.0.weight"), self._ptr(u + ".body.0.bias")
        sw.body2_w, sw.body2_b = self._ptr(u + ".body.2.weight"), self._ptr(u + ".body.2.bias")
        sw.routing_w, sw.routing_b = self._ptr(u + ".routing.0.weight"), self._ptr(u + ".routing.0.bias")
        sw.offset_w, sw.offset_b = self._ptr(u + ".offset.weight"), self._ptr(u + ".offset.bias")
        sw.st_offset_w, sw.st_offset_b = self._ptr(u + ".st_offset.weight"), self._ptr(u + ".st_offset.bias")
        sw.compress, sw.expand = self._ptr(u + ".weight_compress"), self._ptr(u + ".weight_expand")
        self._keep.append(sw)
        H, W = self.H, self.W
        self.rel_y, self.rel_x = self._buf(H), self._buf(W)
        self.base_y, self.base_x = self._buf(H), self._buf(W)
        self.cell_y, self.cell_x = self._buf(H, dtype=torch.int32), self._buf(W, dtype=torch.int32)
        self.corner_y, self.corner_x = self._buf(H, dtype=torch.int32), self._buf(W, dtype=torch.int32)
        self.table = self._buf(H * W, 8)
        # index vectors + per-scale MLP table: input independent, computed once per plan on the device
        K.check(lib.savsr_satu_index(ctx, C.byref(sw), self.h, self.w, H, W, float(self.scale[0]), float(self.scale[1]),
                                     self.rel_y.data_ptr(), self.rel_x.data_ptr(), self.cell_y.data_ptr(), self.cell_x.data_ptr(),
                                     self.base_y.data_ptr(), self.base_x.data_ptr(), self.corner_y.data_ptr(),
                                     self.corner_x.data_ptr(), self.table.data_ptr(), self._stream().cuda_stream))
        tab, by, bx = self.table.data_ptr(), self.base_y.data_ptr(), self.base_x.data_ptr()
        # HR stage + tail in ONE kernel (savsr_arch.py:364-376, 738-739): gathers, routed experts, and -- composed on the host because
        # nothing between them is non-linear -- fusion 128->64 and the 3x3 tail as 27 per-tap partial products per HR pixel, summed
        # over the neighbourhood in shared memory; bias + bilinear skip + fp32 NCHW stores.  No HR-resolution intermediate exists.
        hw = self.store.get(("satu_hr_weights", self.fmt), lambda: satu_hr_pack(satu_hr_compose(P, self.device), self.fmt, self.device))
        zb = self._dev("satu_hr.zbias", lambda: satu_hr_compose(P, self.device)[4])
        tb = self._ptr("tail.bias")
        hwp, outp, cen = hw.data_ptr(), self.out.data_ptr(), t // 2
        hr_flops = 2.0 * B * self.H * self.W * (64 * 32 + 32 * 64 + 128 * 64 + 64 * 3 * 9)      # compress, expand, fusion, tail (reference counts)
        self._emit(lambda st: satu_hr(ctx, lrh, TR, STA, hh, ww, H, W, tab, by, bx, hwp, zb, tb, xin, t, cen, outp, st),
                   kind="satu_hr", flops=hr_flops,
                   rec=lambda cp: add_satu_hr(cp, lrh, TR, STA, hh, ww, H, W, tab, by, bx, hwp, zb, tb, xin, t, cen, outp))
        # declared traffic beyond the compulsory SATU bytes (per sample): only the 16-bit sta intermediate (written by kconv_sta, read here)
        self.satu_extra_bytes_per_sample = 2 * 64 * self.hp * self.wp * 2
        self._stream().synchronize()
        self._pack_src.clear()

    # ------------------------------------------------------------------ execution
    # Every entry point below runs under torch.cuda.device(self.device) and takes the current stream OF THAT DEVICE, so a
    # module on cuda:1 works while the caller's current device is cuda:0 (the C launchers also switch device themselves).
    def _stream(self) -> "torch.cuda.Stream":
        return torch.cuda.current_stream(self.device)

    def run(self) -> None:
        """Launch the whole forward on the device's current stream (x_in -> out)."""
        with torch.cuda.device(self.device), pdl(self.ctx, self.B <= 2):
            self.ctx.set_format(self.fmt)           # the format is context state read at launch (baked into captured graphs)
            st = self._stream().cuda_stream
            if self.cplan is not None:              # the whole list in one C call (savsr_plan_run)
                K.check(self.lib.savsr_plan_run(self.cplan.handle, st))
                return
            for op in self.ops:
                rc = op(st)
                if rc:
                    K.check(rc)

    def run_profiled(self, detail: bool = False) -> Dict[str, Dict[str, float]]:
        """Eager run with a CUDA-event pair around every op on the launching stream.
        Returns {kind: {"ms": total device ms, "flops": algorithmic FLOPs, "ops": count, "launches": kernels}};
        with `detail` the conv kinds are further split by (groups per launch, sources per group, "osa" = per-sample weights)."""
        with torch.cuda.device(self.device):
            self.ctx.set_format(self.fmt)
            stream = self._stream()
            st = stream.cuda_stream
            evs = []
            for op in self.ops:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                rc = op(st)
                e1.record(stream)
                if rc:
                    K.check(rc)
                evs.append((e0, e1))
            stream.synchronize()
        out: Dict[str, Dict[str, float]] = {}
        for (kind, flops, launches, tag), (e0, e1) in zip(self.op_meta, evs):
            d = out.setdefault(f"{kind}:{tag}" if (detail and tag) else kind, dict(ms=0.0, flops=0.0, ops=0, launches=0))
            d["ms"] += e0.elapsed_time(e1); d["flops"] += flops; d["ops"] += 1; d["launches"] += launches
        return out

    def time_ops_graph(self, select: Callable[[str, str], bool], reps: int = 5) -> Dict[str, float]:
        """Device time of a SUBSET of the plan's ops (select(kind, detail)) replayed back to back as their own CUDA graph: the sustained
        per-launch duration of one kernel family under the same conditions as the timed forward (graph launch, power-capped clocks),
        which an eager pass with an event pair around every op does not give (idle gaps between ops let the clocks recover).
        Results are not meaningful (ops run out of program order on whatever the arenas hold); only the timing is used."""
        idx = [i for i, (kind, _, _, detail) in enumerate(self.op_meta) if select(kind, detail)]
        if not idx:
            return dict(ms=0.0, flops=0.0, launches=0, ops=0)
        with torch.cuda.device(self.device):
            self.ctx.set_format(self.fmt)
            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=torch.cuda.Stream(self.device)):
                st = torch.cuda.current_stream(self.device).cuda_stream
                for i in idx:
                    rc = self.ops[i](st)
                    if rc:
                        K.check(rc)
            stream = self._stream()
            g.replay()                                   # warm-up
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(reps):
                g.replay()
            e1.record(stream)
            stream.synchronize()
        return dict(ms=e0.elapsed_time(e1) / reps, flops=sum(self.op_meta[i][1] for i in idx), launches=sum(self.op_meta[i][2] for i in idx), ops=len(idx))

    def capture(self) -> None:
        """Capture run() into a CUDA graph (after one eager warm-up that sets kernel attributes)."""
        if self.graph is not None:
            return
        with torch.cuda.device(self.device):
            self.run()
            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            # an explicit capture stream ON THIS PLAN'S DEVICE: torch's default capture stream is created once per process on
            # whatever device was current then, and capturing through it on another device records an empty graph
            with torch.cuda.graph(g, stream=torch.cuda.Stream(self.device)):
                self.run()
            self.graph = g

    def run_graph(self) -> None:
        if self.graph is None:
            self.capture()
        with torch.cuda.device(self.device):
            self.graph.replay()

    def forward_into(self, x: torch.Tensor, out: torch.Tensor, graph: bool = True) -> None:
        """x -> out through the plan's staging buffers (graph replay reads / writes fixed addresses), all on the device's current
        stream: fp32 [B,7,3,h,w] -> [B,3,H,W], or with io="bgr_u8" uint8 [B,7,h,w,3] -> [B,H,W,3]."""
        if self.io in FRAME_MODES:
            raise ValueError(f'a plan with io="{self.io}" reads frames in place: call forward_frames_into')
        with torch.cuda.device(self.device):
            self.x_in.copy_(x, non_blocking=True)
            if graph:
                self.run_graph()
            else:
                self.run()
            out.copy_(self.out, non_blocking=True)

    def write_frame_table(self, ptrs: Sequence[int]) -> None:
        """Enqueue the writer of the frame table (io="bgr_u8_frames" or "bgr48_frames") on the device's current stream: B*7 device
        addresses of BGR [h,w,3] frames of the mode's sample type, window n = ptrs[7n : 7n + 7].  The addresses travel in the launch
        arguments (savsr_write_frame_table), so nothing waits for the stream; the writer runs in stream order before the forward that reads the table, outside any captured graph."""
        if len(ptrs) != self.frame_table.numel():
            raise ValueError(f"plan built for {self.frame_table.numel()} frame pointers, got {len(ptrs)}")
        arr = (C.c_void_p * len(ptrs))(*ptrs)
        with torch.cuda.device(self.device):
            K.check(self.lib.savsr_write_frame_table(self.ctx.handle, self.frame_table.data_ptr(), arr, len(ptrs), self._stream().cuda_stream))

    def forward_frames_into(self, ptrs: Sequence[int], out: torch.Tensor, graph: bool = True, out_format: Optional[str] = None,
                            out_colorspace: str = "bt601", out_color_range: str = "tv") -> None:
        """io="bgr_u8_frames" or "bgr48_frames": the frames at the B*7 device addresses `ptrs` (see write_frame_table) -> out BGR
        [B,H,W,3] of the mode's sample type, all on the device's current stream.  The frames are read in place by the forward: they must
        stay valid, in stream order, until it has run.  With a YUV out_format of the same depth (4:2:0 or 4:2:2; uint8 or uint16), out is
        [B, *colour.yuv_shape(H, W, out_format)] and the colour conversion reads the output staging buffer in place of the copy
        (colour.bgr_to_yuv, with the matrix out_colorspace and the range out_color_range).  out_format None is the mode's packed
        BGR ("bgr24", "bgr48le"), which takes only the default colour pair: there is nothing to convert."""
        self._forward_table_into(lambda: self.write_frame_table(ptrs), out, graph, out_format, out_colorspace, out_color_range)

    def write_scene_frame_table(self, ring: torch.Tensor, cut: torch.Tensor, first: int, received: int, finished: bool) -> None:
        """Enqueue savsr_write_scene_frame_table on the device's current stream: the table of the B windows of frames first .. first + B - 1
        of a stream whose frame t sits in slot t % R of `ring` (contiguous [R, h, w, 3] of the mode's sample type), each window folded into
        its shot as the device cut flags `cut` (uint8 [R], written by scenes.Detector) mark it.  `received`: frames scored so far;
        `finished`: the stream has ended at `received`.  Nothing is read back: the host does not need to know the cuts."""
        if self.io not in FRAME_MODES:
            raise ValueError(f'write_scene_frame_table needs a plan with io="bgr_u8_frames" or "bgr48_frames", this one has io={self.io!r}')
        if ring.dtype != FRAME_MODES[self.io] or ring.dim() != 4 or tuple(ring.shape[1:]) != (self.h, self.w, 3) or not ring.is_contiguous():
            raise ValueError(f"the ring must be a contiguous {str(FRAME_MODES[self.io]).replace('torch.', '')} tensor [R, {self.h}, {self.w}, 3], "
                             f"got {ring.dtype} {tuple(ring.shape)}")
        if cut.dtype != torch.uint8 or tuple(cut.shape) != (ring.shape[0],):
            raise ValueError(f"cut must be a uint8 tensor [{ring.shape[0]}], got {cut.dtype} {tuple(cut.shape)}")
        fb = self.h * self.w * 3 * ring.element_size()
        with torch.cuda.device(self.device):
            K.check(self.lib.savsr_write_scene_frame_table(self.ctx.handle, self.frame_table.data_ptr(), ring.data_ptr(), fb, ring.shape[0],
                                                            cut.data_ptr(), int(first), self.B, int(received), int(bool(finished)),
                                                            self._stream().cuda_stream))

    def forward_scene_frames_into(self, ring: torch.Tensor, cut: torch.Tensor, first: int, received: int, finished: bool, out: torch.Tensor,
                                  graph: bool = True, out_format: Optional[str] = None, out_colorspace: str = "bt601",
                                  out_color_range: str = "tv") -> None:
        """forward_frames_into with the table written on the device by write_scene_frame_table instead of from host pointers: the windows
        of frames first .. first + B - 1 of the ring, folded at the cuts the device flags mark.  The launch list, the graph and the
        output conversion are those of forward_frames_into."""
        self._forward_table_into(lambda: self.write_scene_frame_table(ring, cut, first, received, finished), out, graph, out_format,
                                 out_colorspace, out_color_range)

    def _forward_table_into(self, write_table: Callable[[], None], out: torch.Tensor, graph: bool, out_format: Optional[str],
                            out_colorspace: str, out_color_range: str) -> None:
        if self.io not in FRAME_MODES:
            raise ValueError(f'forward_frames_into needs a plan with io="bgr_u8_frames" or "bgr48_frames", this one has io={self.io!r}')
        bgr = "bgr48le" if self.io == "bgr48_frames" else "bgr24"
        out_format = bgr if out_format is None else colour.check_format(out_format, "out_format")
        if colour.bgr_format(out_format) != bgr:
            raise ValueError(f'out_format {out_format!r} has another depth than the frames of io="{self.io}" ({bgr})')
        cs = (colour.check_colorspace(out_colorspace, "out_colorspace"), colour.check_color_range(out_color_range, "out_color_range"))
        if out_format == bgr and cs != ("bt601", "tv"):
            raise ValueError(f"out_colorspace / out_color_range {cs} need a YUV out_format: {out_format} output is not converted")
        with torch.cuda.device(self.device):
            write_table()
            if graph:
                self.run_graph()
            else:
                self.run()
            if out_format == bgr:
                out.copy_(self.out, non_blocking=True)
            else:
                colour.bgr_to_yuv(self.out, out_format, out=out, colorspace=cs[0], color_range=cs[1])

    def activation_absmax(self) -> float:
        """Largest |value| currently held anywhere in the LR arena (every trunk activation of the last forward), read in the plan's
        16-bit format.  For the fp16 path: its distance from 65504 is the headroom of that input (SAVSR.forward checks it once per plan)."""
        dt = torch.float16 if self.fmt == K.FMT_FP16 else torch.bfloat16
        with torch.cuda.device(self.device):
            peak = float(torch.linalg.vector_norm(self.arena_lr_t.view(dt).reshape(-1), ord=float("inf")))      # one reduction pass, no temporary
            return peak if peak == peak else float("inf")                                                          # NaN counts as overflow

    def forward_c(self, x: torch.Tensor, out: torch.Tensor) -> None:
        """x -> out through ONE C call (savsr_forward, or savsr_forward_u8 for io="bgr_u8": staging copies + the recorded launch list),
        eagerly on the device's current stream -- what a non-Python host would call.  Shapes and dtypes as in forward_into."""
        if self.cplan is None:
            raise K.SavsrError("this plan has no C-side launch list")
        if self.io in FRAME_MODES:
            raise ValueError(f'a plan with io="{self.io}" reads frames in place: call forward_frames_c')
        u8 = self.io == "bgr_u8"
        dt = torch.uint8 if u8 else torch.float32
        if not (x.is_cuda and out.is_cuda and x.is_contiguous() and out.is_contiguous() and x.dtype == out.dtype == dt):
            raise ValueError(f"savsr_forward{'_u8' if u8 else ''} takes contiguous {'uint8' if u8 else 'fp32'} CUDA tensors")
        if tuple(x.shape) != tuple(self.x_in.shape) or tuple(out.shape) != tuple(self.out.shape):
            raise ValueError(f"plan built for {tuple(self.x_in.shape)} -> {tuple(self.out.shape)}, got {tuple(x.shape)} -> {tuple(out.shape)}")
        fwd = self.lib.savsr_forward_u8 if u8 else self.lib.savsr_forward
        with torch.cuda.device(self.device):
            K.check(fwd(self.cplan.handle, x.data_ptr(), out.data_ptr(), self._stream().cuda_stream))

    def forward_frames_c(self, ptrs: Sequence[int], out: torch.Tensor) -> None:
        """io="bgr_u8_frames" or "bgr48_frames": as forward_frames_into through ONE C call (savsr_forward_u8_frames /
        savsr_forward_u16_frames: table writer + the recorded launch list + the output copy), eagerly on the device's current stream --
        what a non-Python host would call."""
        if self.cplan is None:
            raise K.SavsrError("this plan has no C-side launch list")
        if self.io not in FRAME_MODES:
            raise ValueError(f'forward_frames_c needs a plan with io="bgr_u8_frames" or "bgr48_frames", this one has io={self.io!r}')
        if len(ptrs) != self.frame_table.numel():
            raise ValueError(f"plan built for {self.frame_table.numel()} frame pointers, got {len(ptrs)}")
        dt = FRAME_MODES[self.io]
        name = "savsr_forward_u8_frames" if dt == torch.uint8 else "savsr_forward_u16_frames"
        if not (out.is_cuda and out.is_contiguous() and out.dtype == dt and tuple(out.shape) == tuple(self.out.shape)):
            raise ValueError(f"{name} writes a contiguous {str(dt).replace('torch.', '')} CUDA tensor of shape {tuple(self.out.shape)}")
        arr = (C.c_void_p * len(ptrs))(*ptrs)
        with torch.cuda.device(self.device):
            K.check(getattr(self.lib, name)(self.cplan.handle, arr, out.data_ptr(), self._stream().cuda_stream))

    def release(self) -> None:
        """Drop the CUDA graph and every device buffer now (plan-cache eviction), instead of waiting for the collector."""
        self.graph = None
        self.cplan = None
        self.ops.clear()
        self._keep.clear()
        self._pack_src.clear()
        self.tap_bufs.clear()
        for name in ("arena_lr_t", "x_in", "frame_table", "out", "table", "lr"):
            if hasattr(self, name):
                setattr(self, name, None)
        self.nbytes = 0

    def read_tap(self, name: str) -> torch.Tensor:
        """fp32 NCHW snapshot of a named intermediate requested via `taps` (test / debug only)."""
        return self.tap_bufs[name]
