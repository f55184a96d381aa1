"""Native training step of SAVSR on libsavsr_sm100 (SURVEY.md section 8 row f1, stage B).

The reference trains through autograd: forward, Charbonnier, backward through cuDNN dgrad / wgrad, Adam, EMA
(lbasicsr/models/sr_model.py:101-128, asvsr_model.py:21-29, losses/basic_loss.py:22-24, base_model.py:75-82).  ``TrainPlan`` is
the same step as a STATIC LAUNCH LIST, the way ``engine.Plan`` is for inference: activations AND their gradients live in one
16-bit NHWC arena, every 3x3 / 1x1 convolution of the trunk runs forward, data gradient and weight gradient on the tcgen05
kernels without any layout conversion in between, and the whole step (forward, loss, backward, optimizer) is replayed as CUDA
graphs, one per scale.

  forward   the grouped implicit-GEMM launches of the inference plan (both propagation directions x 3 / 5 streams per launch),
            every activation kept (no slot recycling)
  backward  generated from the forward list in reverse:
              savsr_grad_prep      g = (dV * cscale + cadd) * act'(out)  -> NHWC slot + NCHW T-slot + bias gradient
              savsr_conv           data gradient: the forward kernel on g with transposed, flipped filters; contributions of
                                   several convolutions to one activation are K-stacked into ONE multi-source group
              savsr_conv_wgrad_batched  ALL weight gradients of the step in one persistent launch at the end (the operands stay
                                   alive in the T-arena), except OSA-Conv's per-sample ones, which the attention backward needs early
  weights   one table-driven savsr_pack_conv_chunks launch per step packs every filter in both orientations from the flat fp32
            master copy; Adam + EMA is one kernel over the flat buffers (savsr_adam_ema); data parallelism = one NCCL all-reduce
            of the flat gradient buffer.

  attention OSA-Conv's prologue (pooled means -> scale_routing -> ScaleAttention with BatchNorm on batch statistics -> folded per-sample kernels)
            and its whole backward, the RCAB channel attention, the OSAdapt mask net + combination: native (train_attn.cu, train_mask.cu)

Still on the ATen autograd tape, as ONE "island" between native launches (its inputs / outputs cross as fp32 tensors): SATU at HR resolution
(coordinate MLP, the two gathers, routed experts, fusion), the tail, the bilinear skip and the loss; SATU's per-pixel dynamic filter is a
native op inside it (autograd.sta_lrelu).  `native_attn=False` / `native_mask=False` run the attention MLPs / the mask net as islands too
(cross-checks).  Two ways in: NativeTrainer (the whole step: forward + loss + backward as one CUDA graph per scale, the optimizer as another)
and ModuleTraining (SAVSR.forward in train mode = one autograd node; the caller's loss / optimizer / DDP).  No CPU path.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F

from . import _capi as K
from . import train as T
from .engine import context, get_hw, normalize_scale, pdl

L_ACT = K.ACT_LRELU
MAX_NATIVE_BATCH = 32      # samples per GPU the native attention kernels take (kMaxBatchT, csrc/train_attn.cu); above it they run as ATen islands
CHUNK3 = 9 * 8192          # bytes of the nine [64][64] 16-bit blocks of one (64 x 64 channel) filter corner


def _dev_index(dev: torch.device) -> int:
    if dev.index is not None:
        return dev.index
    return torch.cuda.current_device() if dev.type == "cuda" else 0


def _require_cuda(dev: torch.device) -> None:
    if dev.type != "cuda":
        raise RuntimeError("savsr_b200.trainplan runs on CUDA (sm_100a) only; there is no CPU fallback")


# ====================================================================================================== flat parameters
class FlatParams:
    """The module's parameters re-pointed into ONE flat fp32 buffer, with flat gradient / Adam moment / EMA buffers beside it
    (views keep the reference's names and shapes, so state_dict / load_state_dict / external optimizers keep working)."""

    def __init__(self, module: torch.nn.Module, ema: bool = True, assign_grads: bool = True):
        named = [(n, p) for n, p in module.named_parameters() if p.requires_grad]
        if not named:
            raise ValueError("module has no trainable parameters")
        dev = named[0][1].device
        _require_cuda(dev)
        self.device = dev
        offs, total = {}, 0
        for n, p in named:
            offs[n] = total
            total += (p.numel() + 3) // 4 * 4                 # 16-byte aligned views
        self.n = total
        self.p = torch.zeros(total, device=dev)
        self.g = torch.zeros(total, device=dev)
        self.m = torch.zeros(total, device=dev)
        self.v = torch.zeros(total, device=dev)
        self.P: Dict[str, torch.Tensor] = {}
        self.G: Dict[str, torch.Tensor] = {}
        with torch.no_grad():
            for n, p in named:
                o, k = offs[n], p.numel()
                view = self.p[o:o + k].view(p.shape)
                view.copy_(p.data)
                p.data = view
                gview = self.g[o:o + k].view(p.shape)
                if assign_grads:
                    p.grad = gview
                self.P[n], self.G[n] = p, gview
        self.ema = self.p.clone() if ema else None
        self.offsets = offs
        self.ptrs = [p.data_ptr() for p in self.P.values()]
        self.step_t = torch.zeros(1, device=dev)              # Adam step count as a device scalar (graph replay reads it)

    def intact(self) -> bool:
        """False once something re-allocated the parameters (.to(), .half(), a replaced Parameter): the flat views are then stale."""
        return all(p.data_ptr() == q for p, q in zip(self.P.values(), self.ptrs))

    def ema_view(self, name: str) -> torch.Tensor:
        o, p = self.offsets[name], self.P[name]
        return self.ema[o:o + p.numel()].view(p.shape)

    def view(self, buf: torch.Tensor, name: str) -> torch.Tensor:
        """Parameter `name`'s slice of one of the flat buffers (p, g, m, v, ema), in the parameter's shape."""
        o, p = self.offsets[name], self.P[name]
        return buf[o:o + p.numel()].view(p.shape)


class FlatAdam(torch.optim.Optimizer):
    """Adam + EMA over the flat buffers of `FlatParams` (one savsr_adam_ema launch) as a torch.optim.Optimizer, so that the reference's
    schedulers (torch.optim.lr_scheduler, BasicSR's warm-up / CosineAnnealingRestartLR) drive it and its state_dict is the one
    torch.optim.Adam writes for the same parameters: one group, the module's trainable parameters in named_parameters() order
    (the order of the reference's setup_optimizers), state[i] = {'step', 'exp_avg', 'exp_avg_sq'}.  The moments are views of the flat
    buffers, so state_dict() copies nothing and load_state_dict() copies into them.

    step(): eagerly, savsr_adam_ema with the group's lr; with use_graph, the captured savsr_adam_ema_dev reads the lr from a device
    scalar that is rewritten (one small fill on the current stream) only when the group's lr changed since the last write.  No weight
    decay, no AMSGrad, no maximize: load_state_dict refuses state that asks for them."""

    def __init__(self, flat: FlatParams, ctx: K.Context, lr: float = 2e-4, betas=(0.9, 0.99), eps: float = 1e-8, ema_decay: float = 0.999,
                 world_size: int = 1, use_graph: bool = False):
        defaults = dict(torch.optim.Adam([torch.zeros(1)], lr=lr, betas=betas, eps=eps).defaults)      # torch's group keys, whatever its version
        super().__init__(list(flat.P.values()), defaults)
        self.flat, self.ctx = flat, ctx
        self.names = list(flat.P)
        self.ema_decay, self.world, self.use_graph = ema_decay, world_size, use_graph
        self.lr_dev = torch.full((1,), float(lr), device=flat.device)     # what the captured launch reads
        self._lr_written = float(lr)
        self._graph: Optional[torch.cuda.CUDAGraph] = None
        self._graph_key: Optional[tuple] = None                           # (betas, eps) baked into the captured launch

    @property
    def group(self) -> dict:
        return self.param_groups[0]

    def _hyper(self) -> tuple:
        g = self.group
        if g.get("weight_decay", 0) != 0 or g.get("amsgrad", False) or g.get("maximize", False):
            raise ValueError("the flat Adam kernel implements neither weight decay nor AMSGrad nor maximize")
        return float(g["betas"][0]), float(g["betas"][1]), float(g["eps"])

    def _launch(self, lr_dev: bool) -> None:
        f = self.flat
        b1, b2, eps = self._hyper()
        st = torch.cuda.current_stream(f.device).cuda_stream
        ema = f.ema.data_ptr() if f.ema is not None else None
        f.step_t.add_(1.0)
        if lr_dev:
            K.check(self.ctx.lib.savsr_adam_ema_dev(self.ctx.handle, f.p.data_ptr(), f.g.data_ptr(), f.m.data_ptr(), f.v.data_ptr(), ema, f.n,
                                                    self.lr_dev.data_ptr(), b1, b2, eps, f.step_t.data_ptr(), self.ema_decay, 1.0 / self.world, st))
        else:
            K.check(self.ctx.lib.savsr_adam_ema(self.ctx.handle, f.p.data_ptr(), f.g.data_ptr(), f.m.data_ptr(), f.v.data_ptr(), ema, f.n,
                                                float(self.group["lr"]), b1, b2, eps, f.step_t.data_ptr(), self.ema_decay, 1.0 / self.world, st))

    @torch.no_grad()
    def step(self, closure=None):
        """One Adam + EMA update from the flat gradient buffer (the caller has filled it: NativeTrainer.step does)."""
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        if not self.use_graph:
            self._launch(lr_dev=False)
            return loss
        dev = self.flat.device
        if self._graph is None or self._graph_key != self._hyper():
            og = torch.cuda.CUDAGraph()
            with torch.cuda.graph(og, stream=torch.cuda.Stream(dev)):
                self._launch(lr_dev=True)
            self._graph, self._graph_key = og, self._hyper()           # (capture does not execute: nothing to roll back)
        lr = float(self.group["lr"])
        if lr != self._lr_written:
            self.lr_dev.fill_(lr)
            self._lr_written = lr
        self._graph.replay()
        return loss

    def zero_grad(self, set_to_none: bool = True) -> None:
        """The gradients are views of the flat gradient buffer and stay so: zero it (set_to_none is ignored)."""
        self.flat.g.zero_()

    # ---- checkpoints: the layout of torch.optim.Adam.state_dict()
    def state_dict(self) -> dict:
        f = self.flat
        step = float(f.step_t.item())
        self.state.clear()
        if step > 0:
            for n, p in f.P.items():
                self.state[p] = {"step": torch.tensor(step, dtype=torch.float32), "exp_avg": f.view(f.m, n), "exp_avg_sq": f.view(f.v, n)}
        try:
            return super().state_dict()
        finally:
            self.state.clear()

    def load_state_dict(self, state_dict: dict) -> None:
        """Take over a state written by FlatAdam or torch.optim.Adam for the same parameters: moments, step, the group's lr / initial_lr /
        betas / eps.  Raises ValueError on what the kernel cannot continue (several groups, other parameters, per-parameter step
        counts, weight decay, AMSGrad, maximize)."""
        groups = state_dict.get("param_groups", [])
        if len(groups) != 1:
            raise ValueError(f"FlatAdam holds one parameter group; the state has {len(groups)}")
        saved = groups[0]
        if saved.get("weight_decay", 0) != 0:
            raise ValueError(f"weight_decay={saved['weight_decay']} is not implemented by the flat Adam kernel (it needs 0)")
        for key in ("amsgrad", "maximize"):
            if saved.get(key, False):
                raise ValueError(f"{key}=True is not implemented by the flat Adam kernel")
        f = self.flat
        ids = list(saved["params"])
        if len(ids) != len(self.names):
            raise ValueError(f"the state holds {len(ids)} parameters, this optimizer {len(self.names)}")
        st = state_dict.get("state", {})
        steps = set()
        for pid, n in zip(ids, self.names):
            s = st.get(pid)
            if s is None:
                steps.add(0.0)
                continue
            steps.add(float(s["step"]))
            for key in ("exp_avg", "exp_avg_sq"):
                if tuple(s[key].shape) != tuple(f.P[n].shape):
                    raise ValueError(f"parameter {pid} ({n}): {key} has shape {tuple(s[key].shape)}, the parameter {tuple(f.P[n].shape)}")
        if len(steps) > 1:
            raise ValueError(f"the parameters have different step counts {sorted(steps)}; the flat kernel keeps one")
        with torch.no_grad():
            for pid, n in zip(ids, self.names):
                s = st.get(pid)
                for buf, key in ((f.m, "exp_avg"), (f.v, "exp_avg_sq")):
                    if s is None:
                        f.view(buf, n).zero_()
                    else:
                        f.view(buf, n).copy_(s[key])
            f.step_t.fill_(steps.pop() if steps else 0.0)
        group = {k: v for k, v in saved.items() if k != "params"}      # as torch's load_state_dict: the saved group with our parameters
        for k, v in self.defaults.items():
            group.setdefault(k, v)
        group["params"] = self.group["params"]
        self.param_groups[0] = group
        self.state.clear()
        if self._graph is not None and self._graph_key != self._hyper():
            self._graph = None                                          # betas / eps are baked into the captured launch


# ====================================================================================================== packed weights
class TrainWeights:
    """Packed tensor-core copies of every trunk filter, forward orientation and transposed / flipped (data gradient), refreshed
    from the flat fp32 master weights by ONE table-driven launch per step.  Shared by all plans (scales) of one module."""

    def __init__(self, flat: FlatParams, ctx: K.Context):
        self.flat, self.ctx, self.lib = flat, ctx, ctx.lib
        self.dev = flat.device
        self.chunks: List[K.PackChunk] = []
        self._bufs: Dict[tuple, torch.Tensor] = {}
        self._keep: List[object] = []
        self.table: Optional[torch.Tensor] = None
        self.table_count = 0
        self.capacity = 8192
        self.table_dev = torch.zeros(self.capacity * C.sizeof(K.PackChunk), dtype=torch.uint8, device=self.dev)
        # first-layer filters zero-expanded to the packed-frames slot (engine.Plan does the same for inference)
        self.expanded: Dict[tuple, torch.Tensor] = {}
        self.expanded_grad: Dict[tuple, torch.Tensor] = {}
        self._stage_dst: List[torch.Tensor] = []
        self._stage_src: List[torch.Tensor] = []
        self._scatter_dst: List[torch.Tensor] = []
        self._scatter_src: List[torch.Tensor] = []
        self.scratch_grads: List[torch.Tensor] = []

    # ---- registration (plan build time)
    def _chunk(self, w: torch.Tensor, dst_ptr: int, co: int, ci: int, o_base: int, i_base: int, ksize: int, transposed: int) -> None:
        ch = K.PackChunk()
        ch.w, ch.dst = w.data_ptr(), dst_ptr
        ch.co_total, ch.ci_total, ch.o_base, ch.i_base, ch.ksize, ch.transposed = co, ci, o_base, i_base, ksize, transposed
        if len(self.chunks) >= self.capacity:
            raise K.SavsrError("TrainWeights: chunk table full")
        self.chunks.append(ch)
        self.table = None

    def _weight_of(self, key) -> torch.Tensor:
        return self.expanded[key] if isinstance(key, tuple) else self.flat.P[key]

    def fwd(self, key, half: int = 0) -> int:
        """Packed forward operand of parameter `key` ([co][ci][k][k]); returns the pointer of the 64-output-channel block `half`."""
        w = self._weight_of(key)
        co, ci, ks, _ = w.shape
        nsrc, taps = ci // 64, ks * ks
        bk = ("fwd", key)
        if bk not in self._bufs:
            buf = torch.zeros(co * ci * taps * 2, dtype=torch.uint8, device=self.dev)
            self._bufs[bk] = buf
            for ng in range(co // 64):
                for s in range(nsrc):
                    self._chunk(w, buf.data_ptr() + (ng * nsrc + s) * taps * 8192, co, ci, ng * 64, s * 64, ks, 0)
        return self._bufs[bk].data_ptr() + half * nsrc * taps * 8192

    def dgrad(self, stack: Tuple[tuple, ...]) -> int:
        """Data-gradient operand for ONE destination activation: `stack` = ((weight key, source index s, output half h), ...), one
        entry per gradient that flows into it; the transposed chunks are laid out as the K blocks of one multi-source group."""
        bk = ("dgrad", stack)
        if bk not in self._bufs:
            ks = self._weight_of(stack[0][0]).shape[-1]
            taps = ks * ks
            buf = torch.zeros(len(stack) * taps * 8192, dtype=torch.uint8, device=self.dev)
            self._bufs[bk] = buf
            for j, (key, s, h) in enumerate(stack):
                w = self._weight_of(key)
                co, ci = w.shape[0], w.shape[1]
                self._chunk(w, buf.data_ptr() + j * taps * 8192, co, ci, h * 64, s * 64, ks, 1)
        return self._bufs[bk].data_ptr()

    def expand_first_layer(self, prefix: str, which: str, centre: int) -> tuple:
        """conv_c (3 -> 64) / conv_sup (6 -> 64) of savsr_arch.py:456-457 as a [64][64][3][3] filter over the packed-frames slot
        (channel 3 f + c = frame f, colour c).  Staged from the real parameter before every pack; its gradient is scattered back."""
        key = (prefix, which, centre)
        if key in self.expanded:
            return key
        wz = torch.zeros(64, 64, 3, 3, device=self.dev)
        gz = torch.zeros(64, 64, 3, 3, device=self.dev)
        self.expanded[key], self.expanded_grad[key] = wz, gz
        self.scratch_grads.append(gz)
        name = f"{prefix}.{which}.weight"
        P, G = self.flat.P[name], self.flat.G[name]
        c = centre
        pieces = [(3 * c, 0)] if which == "conv_c" else [(3 * (c - 1), 0), (3 * (c + 1), 3)]
        for dst0, src0 in pieces:
            self._stage_dst.append(wz[:, dst0:dst0 + 3]); self._stage_src.append(P.detach()[:, src0:src0 + 3])
            self._scatter_dst.append(G[:, src0:src0 + 3]); self._scatter_src.append(gz[:, dst0:dst0 + 3])
        return key

    def scratch_grad(self, key, shape, scatter_to: Optional[torch.Tensor] = None, rows: Optional[int] = None) -> torch.Tensor:
        """A zero-per-step fp32 gradient staging buffer shared by all plans (keyed); its first `rows` rows are added to `scatter_to`
        after the backward (the tensor-core weight gradient always writes 64 output-channel rows)."""
        k = ("scratch", key)
        if k not in self._bufs:
            buf = torch.zeros(*shape, device=self.dev)
            self._bufs[k] = buf
            self.scratch_grads.append(buf)
            if scatter_to is not None:
                self._scatter_dst.append(scatter_to)
                self._scatter_src.append(buf[:rows] if rows is not None else buf)
        return self._bufs[k]

    # ---- per step
    def finalize(self) -> None:
        if self.table is not None:
            return
        arr = (K.PackChunk * len(self.chunks))(*self.chunks)
        host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8)
        self.table_dev[:host.numel()].copy_(host)
        self.table = self.table_dev
        self.table_count = len(self.chunks)

    def pack(self, st: int) -> None:
        """Stage the expanded first-layer filters and pack every registered chunk (one launch)."""
        self.finalize()
        if self._stage_dst:
            torch._foreach_copy_(self._stage_dst, self._stage_src)
        K.check(self.lib.savsr_pack_conv_chunks(self.ctx.handle, self.table_dev.data_ptr(), 0, self.table_count, st))

    def zero_scratch(self) -> None:
        if self.scratch_grads:
            torch._foreach_zero_(self.scratch_grads)

    def scatter_expanded_grads(self) -> None:
        if self._scatter_dst:
            torch._foreach_add_(self._scatter_dst, self._scatter_src)


# ====================================================================================================== plan
class _Spec:
    """One convolution of a grouped forward launch."""
    __slots__ = ("src", "dst", "wkey", "half", "bias", "act", "slope", "res1", "pool", "src_channels", "osa", "ksize")

    def __init__(self, src, dst, wkey=None, half=0, bias=None, act=K.ACT_NONE, slope=0.2, res1=-1, pool=None, src_channels=0,
                 osa=None, ksize=3):
        self.src, self.dst, self.wkey, self.half, self.bias = list(src), dst, wkey, half, bias
        self.act, self.slope, self.res1, self.pool, self.src_channels, self.osa, self.ksize = act, slope, res1, pool, src_channels, osa, ksize


class _Osa:
    """State of one OSA-Conv (savsr_arch.py:139-172) inside a plan: pooled means -> scale_routing -> ScaleAttention (train-mode
    BatchNorm) -> per-sample folded kernels in both operand orientations, and the buffers of its backward."""

    def __init__(self, plan: "TrainPlan", prefix: str, srcs: Sequence[int], pools: Sequence[torch.Tensor]):
        self.prefix, self.srcs, self.pools = prefix, list(srcs), list(pools)
        B, dev = plan.B, plan.device
        self.ci = 64 * len(srcs)
        self.nsrc = len(srcs)
        ci = self.ci
        self.dwfold = torch.zeros(B, 64, ci, 3, 3, device=dev)     # native attention: used as [B][9 taps][ci][64] (K.WGRAD_TIO)
        self.dpool = torch.zeros(B, ci, device=dev)
        self.packed_fwd = torch.zeros(B * self.nsrc * CHUNK3, dtype=torch.uint8, device=dev)      # [n][s][9][64][64]
        self.packed_bwd = torch.zeros(self.nsrc * B * CHUNK3, dtype=torch.uint8, device=dev)      # [s][n][9][64][64]
        self.fwd_stride = self.nsrc * CHUNK3
        a = prefix + ".attention"
        names = [prefix + ".weight"] + [f"{prefix}.scale_routing.{i}.{k}" for i in (0, 2) for k in ("weight", "bias")]
        names += [a + ".fc.weight", a + ".bn.weight", a + ".bn.bias"] + [f"{a}.{hd}.{k}" for hd in ("channel_fc", "filter_fc", "spatial_fc", "kernel_fc")
                                                                          for k in ("weight", "bias")]
        self.param_names = names
        if plan.native_attn:
            P, G, Bf = plan.P, plan.G, plan.net.B
            lib = plan.lib
            self.scratch = torch.zeros(B, 5 * ci + 192, device=dev)
            self.state = torch.zeros(int(lib.savsr_osa_train_state_floats(B)), device=dev)
            self.datt = torch.zeros(B, ci + 64 + 17, device=dev)
            self.dvec = torch.zeros(int(lib.savsr_osa_train_dvec_floats(B, ci)), device=dev)
            o = K.OsaParams()
            o.ci, o.co, o.att = ci, 64, max(int(ci * 0.0625), 16)
            o.bank = P[prefix + ".weight"].data_ptr()
            o.r0_w, o.r0_b = P[prefix + ".scale_routing.0.weight"].data_ptr(), P[prefix + ".scale_routing.0.bias"].data_ptr()
            o.r2_w, o.r2_b = P[prefix + ".scale_routing.2.weight"].data_ptr(), P[prefix + ".scale_routing.2.bias"].data_ptr()
            o.fc_w = P[a + ".fc.weight"].data_ptr()
            o.bn_scale = o.bn_shift = None
            o.ch_w, o.ch_b = P[a + ".channel_fc.weight"].data_ptr(), P[a + ".channel_fc.bias"].data_ptr()
            o.fl_w, o.fl_b = P[a + ".filter_fc.weight"].data_ptr(), P[a + ".filter_fc.bias"].data_ptr()
            o.sp_w, o.sp_b = P[a + ".spatial_fc.weight"].data_ptr(), P[a + ".spatial_fc.bias"].data_ptr()
            o.kn_w, o.kn_b = P[a + ".kernel_fc.weight"].data_ptr(), P[a + ".kernel_fc.bias"].data_ptr()
            for i, pp in enumerate(pools):
                o.pool[i] = pp.data_ptr()
            o.scratch, o.packed = self.scratch.data_ptr(), self.packed_fwd.data_ptr()
            t = K.OsaTrain()
            t.bn_weight, t.bn_bias = P[a + ".bn.weight"].data_ptr(), P[a + ".bn.bias"].data_ptr()
            t.running_mean, t.running_var = Bf[a + ".bn.running_mean"].data_ptr(), Bf[a + ".bn.running_var"].data_ptr()
            t.momentum, t.eps = T.BN_MOMENTUM, T.BN_EPS
            t.state, t.packed_t = self.state.data_ptr(), self.packed_bwd.data_ptr()
            g = K.OsaGrads()
            g.dwfold, g.d_bank = self.dwfold.data_ptr(), G[prefix + ".weight"].data_ptr()
            g.d_r0_w, g.d_r0_b = G[prefix + ".scale_routing.0.weight"].data_ptr(), G[prefix + ".scale_routing.0.bias"].data_ptr()
            g.d_r2_w, g.d_r2_b = G[prefix + ".scale_routing.2.weight"].data_ptr(), G[prefix + ".scale_routing.2.bias"].data_ptr()
            g.d_fc_w, g.d_bn_w, g.d_bn_b = G[a + ".fc.weight"].data_ptr(), G[a + ".bn.weight"].data_ptr(), G[a + ".bn.bias"].data_ptr()
            g.d_ch_w, g.d_ch_b = G[a + ".channel_fc.weight"].data_ptr(), G[a + ".channel_fc.bias"].data_ptr()
            g.d_fl_w, g.d_fl_b = G[a + ".filter_fc.weight"].data_ptr(), G[a + ".filter_fc.bias"].data_ptr()
            g.d_sp_w, g.d_sp_b = G[a + ".spatial_fc.weight"].data_ptr(), G[a + ".spatial_fc.bias"].data_ptr()
            g.d_kn_w, g.d_kn_b = G[a + ".kernel_fc.weight"].data_ptr(), G[a + ".kernel_fc.bias"].data_ptr()
            g.datt, g.dvec, g.dpool = self.datt.data_ptr(), self.dvec.data_ptr(), self.dpool.data_ptr()
            self.params, self.extra, self.grads = o, t, g
            nbt = a + ".bn.num_batches_tracked"
            if nbt in Bf:
                plan.nbt_counts[nbt] = plan.nbt_counts.get(nbt, 0) + 1
        else:
            self.wfold = torch.zeros(B, 64, ci, 3, 3, device=dev)
            self.chunk_first = len(plan.chunks)
            for n in range(B):
                for s in range(self.nsrc):
                    plan._chunk(self.wfold[n], self.packed_fwd.data_ptr() + (n * self.nsrc + s) * CHUNK3, 64, ci, 0, s * 64, 3, 0)
                    plan._chunk(self.wfold[n], self.packed_bwd.data_ptr() + (s * B + n) * CHUNK3, 64, ci, 0, s * 64, 3, 1)
            self.chunk_count = len(plan.chunks) - self.chunk_first
            self.graph_out = None
            self.leaf = None


class TrainPlan:
    """Forward + backward launch list of one (batch, h, w, scale).  h and w must be even (the training crops are 64 x 64)."""

    def __init__(self, module: torch.nn.Module, flat: FlatParams, weights: TrainWeights, batch: int, h: int, w: int, scale,
                 precision: str = "bf16", native_attn: bool = True, native_mask: bool = True, own_loss: bool = True):
        device = flat.device
        self.own_loss = own_loss                            # False: the caller computes the loss from the returned output and passes its gradient back
        self.dsr: Optional[torch.Tensor] = None
        self.native_attn = native_attn and batch <= MAX_NATIVE_BATCH      # False: the attention MLPs run as ATen islands (cross-check / larger batches)
        self.native_mask = native_mask                      # False: the OSAdapt mask net + combination run as an ATen island (cross-check)
        self._mask_scratch: Optional[dict] = None
        self.nbt_counts: Dict[str, int] = {}
        if h % 2 or w % 2 or h < 2 or w < 2:
            raise ValueError(f"TrainPlan needs even LR sizes >= 2 (training crops), got {h}x{w}")
        if precision != "bf16":
            raise ValueError("the native training step stores gradients in bf16 (fp16 would need loss scaling); precision must be 'bf16'")
        self.module, self.flat, self.W = module, flat, weights
        self.device = device
        self.ctx = context(_dev_index(device))
        self.lib = self.ctx.lib
        self.fmt = K.FMT_BF16
        self.B, self.h, self.w = batch, h, w
        self.scale = normalize_scale(scale)
        self.H, self.Wd = get_hw(h, w, self.scale)
        self.pitch = (w + 7) // 8 * 8
        self.npix = h * w
        self.net = T._Net(module, True)
        self.P, self.G = flat.P, flat.G
        self._keep: List[object] = []
        self.fwd_ops: List[Callable[[int], None]] = []
        self.bwd_ops: List[Callable[[int], None]] = []
        self._builders: List[Callable[[], None]] = []
        self._emit_to = self.fwd_ops
        self.n_slots = 0
        self.n_tslots = 0
        self.gmap: Dict[int, int] = {}
        self.shared: set = set()              # gradient slots aliased by several activations: never modified in place by grad_prep
        self.noreq: set = set()
        self.prep_mod: Dict[int, dict] = {}   # activation slot -> cscale / cadd modifiers of its gradient
        self.gt_of: Dict[int, int] = {}       # conv output slot -> T-slot of its transposed gradient
        self.x3_of: Dict[int, int] = {}       # activation slot -> first of its three shifted T-slots
        self.x3_emitted: set = set()
        self.x3_ops: List[Callable[[int], None]] = []   # run on a side stream, concurrently with the loss island
        self._side: Optional[torch.cuda.Stream] = None
        self.chunks: List[K.PackChunk] = []   # plan-local pack chunks (per-sample OSA kernels)
        self.witems: List[K.WgradItem] = []
        self.deferred: List[int] = []         # indices into witems, run by the final batched launch
        self.launches = {"fwd": 0, "bwd": 0}
        self.kinds: Dict[int, str] = {}
        self.arena: Optional[K.Arena] = None
        self.loss: Optional[torch.Tensor] = None
        with torch.cuda.device(device):
            self.ctx.set_format(self.fmt)
            self._build()

    # ------------------------------------------------------------------ small helpers
    def _new_slot(self) -> int:
        self.n_slots += 1
        return self.n_slots - 1

    def _new_tslots(self, k: int = 1) -> int:
        t = self.n_tslots
        self.n_tslots += k
        return t

    def _emit(self, fn: Callable[[int], None], launches: int = 1, kind: str = "other") -> None:
        self._emit_to.append(fn)
        phase = "fwd" if self._emit_to is self.fwd_ops else "bwd"
        self.kinds[id(fn)] = f"{phase}:{kind}"
        self.launches[phase] += launches

    def _chunk(self, w: torch.Tensor, dst_ptr: int, co: int, ci: int, o_base: int, i_base: int, ksize: int, transposed: int) -> None:
        ch = K.PackChunk()
        ch.w, ch.dst = w.data_ptr(), dst_ptr
        ch.co_total, ch.ci_total, ch.o_base, ch.i_base, ch.ksize, ch.transposed = co, ci, o_base, i_base, ksize, transposed
        self.chunks.append(ch)

    def _buf(self, *shape, dtype=torch.float32) -> torch.Tensor:
        t = torch.zeros(*shape, dtype=dtype, device=self.device)
        self._keep.append(t)
        return t

    def _ah(self):
        return self.arena.handle

    def _gdst(self, slot: int) -> Tuple[int, int]:
        """(dst, res1) for a gradient contribution to activation `slot`: the first one writes, later ones accumulate in place."""
        if slot in self.gmap:
            g = self.gmap[slot]
            if g in self.shared:                        # aliased with another activation's gradient: give this one its own copy first
                own = self._new_slot()
                self._axpby([(own, g, -1, 1.0, 0.0)])
                self.gmap[slot] = own
                g = own
            return g, g
        g = self._new_slot()
        self.gmap[slot] = g
        return g, -1

    # ------------------------------------------------------------------ native launch emitters
    def _axpby(self, entries: Sequence[Tuple[int, int, int, float, float]]) -> None:
        for i in range(0, len(entries), K.MAX_TRAIN_ENTRIES):
            part = entries[i:i + K.MAX_TRAIN_ENTRIES]
            arr = (K.Axpby * len(part))()
            for e, (d, x, y, a, b) in zip(arr, part):
                e.dst_slot, e.x_slot, e.y_slot, e.alpha, e.beta = d, x, y, a, b
            self._keep.append(arr)
            lib, ctx, n = self.lib, self.ctx.handle, len(part)
            self._emit(lambda st, arr=arr, n=n: K.check(lib.savsr_slot_axpby(ctx, self._ah(), arr, n, st)), kind="axpby")

    def _accumulate(self, pairs: Sequence[Tuple[int, int]], scale: float = 1.0) -> None:
        """grad(target) += scale * slot for (target activation, gradient slot) pairs, batched into one launch."""
        ent = []
        for tgt, gslot in pairs:
            if tgt in self.noreq:
                continue
            d, r = self._gdst(tgt)
            ent.append((d, gslot, r, scale, 1.0))
        if ent:
            self._axpby(ent)

    def _conv_launch(self, groups: Sequence[K.ConvGroup], ksize: int = 3) -> None:
        for i in range(0, len(groups), K.MAX_GROUPS):
            part = groups[i:i + K.MAX_GROUPS]
            arr = (K.ConvGroup * len(part))(*part)
            self._keep.append(arr)
            lib, ctx, n = self.lib, self.ctx.handle, len(part)
            self._emit(lambda st, arr=arr, n=n: K.check(lib.savsr_conv(ctx, self._ah(), arr, n, ksize, 64, K.DST_ARENA, K.IMPL_HALO, st)), kind=f"conv{ksize}")

    @staticmethod
    def _group(src: Sequence[int], dst: int, weight: int, bias: int = 0, act: int = K.ACT_NONE, slope: float = 0.2, res1: int = -1,
               wstride: int = 0, pool: int = 0, src_channels: int = 0) -> K.ConvGroup:
        g = K.ConvGroup()
        for i, s in enumerate(src):
            g.src_slot[i] = s
        g.nsrc = len(src)
        g.dst_slot, g.res1_slot, g.res2_slot, g.res2_scale = dst, res1, -1, 0.0
        g.act, g.slope = act, slope
        g.weight, g.weight_sample_stride = weight, wstride
        g.bias, g.mask, g.pool, g.aux_dst = bias or None, None, pool or None, None
        g.src_channels = src_channels
        return g

    def _x3(self, slots: Sequence[int]) -> None:
        """The weight gradient needs these activations as three x-shifted NCHW copies.  The copies depend on the FORWARD only, so
        they are not part of the backward chain: all of them run on a side stream that forks before the loss island and joins
        before the backward starts (TrainPlan.run), i.e. they cost nothing on the critical path."""
        ent = []
        for s in slots:
            if s in self.x3_emitted:
                continue
            self.x3_emitted.add(s)
            if s not in self.x3_of:
                self.x3_of[s] = self._new_tslots(3)
            ent.append((s, self.x3_of[s]))
        for i in range(0, len(ent), K.MAX_TRAIN_ENTRIES):
            part = ent[i:i + K.MAX_TRAIN_ENTRIES]
            arr = (K.Nchw3 * len(part))()
            for e, (s, t) in zip(arr, part):
                e.x_slot, e.t_slot = s, t
            self._keep.append(arr)
            lib, ctx, n = self.lib, self.ctx.handle, len(part)
            fn = lambda st, arr=arr, n=n: K.check(lib.savsr_slot_to_nchw3(ctx, self._ah(), self.tarena.data_ptr(), self.n_tslots, self.pitch, arr, n, st))  # noqa: E731
            self.x3_ops.append(fn)
            self.kinds[id(fn)] = "side:nchw3"
            self.launches["bwd"] += 1

    def _wgrad_launch(self, first: int, count: int) -> None:
        lib, ctx = self.lib, self.ctx.handle
        self._emit(lambda st: K.check(lib.savsr_conv_wgrad_batched(ctx, self.tarena.data_ptr(), self.n_tslots, self.B, self.h, self.w, self.pitch,
                                                                   self.witems_dev.data_ptr(), first, count, st)), kind="wgrad")

    # ------------------------------------------------------------------ convolution: forward + backward builder
    def _weight_ptr(self, sp: _Spec) -> Tuple[int, int]:
        if sp.osa is not None:
            return sp.osa.packed_fwd.data_ptr(), sp.osa.fwd_stride
        return self.W.fwd(sp.wkey, sp.half), 0

    def _conv(self, specs: Sequence[_Spec], ksize: int = 3) -> None:
        groups = []
        for sp in specs:
            assert sp.res1 < 0 or sp.act == K.ACT_NONE, "a fused residual hides the sign of the activation: emit an explicit add"
            wp, ws = self._weight_ptr(sp)
            bias = 0
            if sp.bias is not None:
                bias = self.P[sp.bias].data_ptr() + sp.half * 64 * 4
            groups.append(self._group(sp.src, sp.dst, wp, bias, sp.act, sp.slope, sp.res1, ws, sp.pool.data_ptr() if sp.pool is not None else 0,
                                      sp.src_channels))
        self._conv_launch(groups, ksize)
        specs = list(specs)
        self._builders.append(lambda: self._conv_backward(specs, ksize))

    def _conv_backward(self, specs: Sequence[_Spec], ksize: int) -> None:
        live = [sp for sp in specs if sp.dst in self.gmap]
        if not live:
            return
        # 1. gradient entering each convolution (activation derivative, channel scale, pooled-mean gradient), its transposed copy, bias gradient
        prep = []
        gslot: Dict[int, int] = {}
        for sp in live:
            dv = self.gmap[sp.dst]
            mod = self.prep_mod.get(sp.dst, {})
            identity = sp.act == K.ACT_NONE and not mod
            if identity:
                g = dv
                store = -1
            elif dv in self.shared:
                g = store = self._new_slot()
            else:
                g = store = dv
            gslot[sp.dst] = g
            gt = self._new_tslots(1)
            self.gt_of[sp.dst] = gt
            e = K.GradPrep()
            e.dv_slot, e.out_slot, e.g_slot, e.gt_tslot = dv, sp.dst, store, gt
            e.act, e.slope = sp.act, sp.slope
            cs = mod.get("cscale")
            e.cscale, e.cscale_stride = (cs[0], cs[1]) if cs else (None, 0)
            ca = mod.get("cadd")
            e.cadd, e.cadd_stride, e.cadd_mul = (ca[0], ca[1], ca[2]) if ca else (None, 0, 0.0)
            e.dbias = (self.G[sp.bias].data_ptr() + sp.half * 64 * 4) if sp.bias is not None else None
            prep.append(e)
        for i in range(0, len(prep), K.MAX_TRAIN_ENTRIES):
            part = prep[i:i + K.MAX_TRAIN_ENTRIES]
            arr = (K.GradPrep * len(part))(*part)
            self._keep.append(arr)
            lib, ctx, n = self.lib, self.ctx.handle, len(part)
            self._emit(lambda st, arr=arr, n=n: K.check(lib.savsr_grad_prep(ctx, self._ah(), self.tarena.data_ptr(), self.n_tslots, self.pitch, arr, n, st)), kind="grad_prep")
        # 2. fused residuals (act NONE only): d res1 += g
        self._accumulate([(sp.res1, gslot[sp.dst]) for sp in live if sp.res1 >= 0])
        # 3. data gradients: contributions to one activation from the shared-weight convs of this launch are K-stacked
        stacked: Dict[int, List[Tuple[int, tuple]]] = {}
        per_sample: List[Tuple[int, int, _Spec, int]] = []
        for sp in live:
            for s, tgt in enumerate(sp.src):
                if tgt in self.noreq:
                    continue
                if sp.osa is not None:
                    per_sample.append((tgt, gslot[sp.dst], sp, s))
                else:
                    stacked.setdefault(tgt, []).append((gslot[sp.dst], (sp.wkey, s, sp.half)))
        by_nsrc: Dict[int, List[K.ConvGroup]] = {}
        for tgt, contribs in stacked.items():
            for i in range(0, len(contribs), K.MAX_SRC):
                part = contribs[i:i + K.MAX_SRC]
                wp = self.W.dgrad(tuple(c[1] for c in part))
                d, r = self._gdst(tgt)
                by_nsrc.setdefault(len(part), []).append(self._group([c[0] for c in part], d, wp, res1=r))
                if i + K.MAX_SRC < len(contribs):      # more than five contributions: the next group accumulates, so it needs its own launch
                    self._conv_launch(by_nsrc.pop(len(part)), ksize)
        for n in sorted(by_nsrc):
            self._conv_launch(by_nsrc[n], ksize)
        seen: set = set()
        batch: List[K.ConvGroup] = []
        for tgt, g, sp, s in per_sample:
            if tgt in seen:                            # two per-sample contributions to one activation must not share a launch
                self._conv_launch(batch, ksize)
                batch, seen = [], set()
            seen.add(tgt)
            d, r = self._gdst(tgt)
            batch.append(self._group([g], d, sp.osa.packed_bwd.data_ptr() + s * self.B * CHUNK3, res1=r, wstride=CHUNK3))
        if batch:
            self._conv_launch(batch, ksize)
        # 4. weight gradients: table items, deferred to the final batched launch (OSA-Conv: right away, its fold backward needs them)
        inline: List[int] = []
        for sp in live:
            for s, src in enumerate(sp.src):
                it = K.WgradItem()
                it.g_tslot = self.gt_of[sp.dst]
                it.ksize = ksize
                if sp.osa is not None:
                    it.dw, it.ci_total, it.ci_off, it.o_off = sp.osa.dwfold.data_ptr(), sp.osa.ci, s * 64, 0
                    it.per_sample, it.sample_stride = 1, 64 * sp.osa.ci * 9
                    it.layout = K.WGRAD_TIO if self.native_attn else K.WGRAD_OIHW      # [tap][i][o] for the native fold backward (vector atomics)
                else:
                    wt = self.W.expanded_grad[sp.wkey] if isinstance(sp.wkey, tuple) else self.G[sp.wkey]
                    it.dw, it.ci_total, it.ci_off, it.o_off = wt.data_ptr(), wt.shape[1], s * 64, sp.half * 64
                    it.per_sample, it.sample_stride = 0, 0
                self._wsrc.append(src)
                self.witems.append(it)
                (inline if sp.osa is not None else self.deferred).append(len(self.witems) - 1)
        if inline:
            self._x3([self._wsrc[i] for i in inline])
            assert inline == list(range(inline[0], inline[0] + len(inline)))
            first, count = inline[0], len(inline)
            self._wgrad_launch(first, count)

    # ------------------------------------------------------------------ explicit residual add
    def _add(self, triples: Sequence[Tuple[int, int, int]]) -> None:
        """out = x + a for (out, x, a) triples in one launch; backward: grad(a) aliases grad(out), grad(x) += grad(out)."""
        self._axpby([(o, x, a, 1.0, 1.0) for o, x, a in triples])
        triples = list(triples)

        def bwd():
            pairs = []
            for o, x, a in triples:
                if o not in self.gmap:
                    continue
                g = self.gmap[o]
                self.gmap[a] = g
                self.shared.add(g)
                pairs.append((x, g))
            self._accumulate(pairs)
        self._builders.append(bwd)

    # ------------------------------------------------------------------ islands (ATen autograd between native launches)
    def _export(self, slot: int) -> torch.Tensor:
        out = torch.empty(self.B, 64, self.h, self.w, device=self.device)
        K.check(self.lib.savsr_arena_export(self._ah(), slot, out.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream))
        return out

    def _import(self, slot: int, t: torch.Tensor) -> None:
        t = t.contiguous()
        self._keep_step.append(t)
        K.check(self.lib.savsr_arena_import(self._ah(), slot, t.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream))

    def _import_grads(self, pairs: Sequence[Tuple[int, Callable[[], torch.Tensor]]]) -> None:
        """Backward-program ops that bring island gradients (fp32 NCHW, fetched lazily at run time) into the gradient slots."""
        acc = []
        for tgt, fetch in pairs:
            if tgt in self.noreq:
                continue
            tmp = self._new_slot()
            self._emit(lambda st, tmp=tmp, fetch=fetch: self._import(tmp, fetch()), kind="import")
            acc.append((tgt, tmp))
        self._accumulate(acc)

    def _param_grads(self, names: Sequence[str], grads: Sequence[Optional[torch.Tensor]]) -> None:
        dst, src = [], []
        for n, g in zip(names, grads):
            if g is not None:
                dst.append(self.G[n]); src.append(g)
        if dst:
            torch._foreach_add_(dst, src)

    def _osa_fold(self, o: _Osa) -> None:
        """Forward island of one OSA-Conv: pooled means -> scale_routing -> ScaleAttention (train-mode BatchNorm) -> folded kernels."""
        net, B, pre = self.net, self.B, o.prefix

        def fwd(st):
            pooled = torch.cat([p.sum(1) for p in o.pools], 1) / float(self.npix)
            o.leaf = pooled.detach().requires_grad_(True)
            with torch.enable_grad():
                o.graph_out = T.osa_fold(net, pre, o.leaf, self.scale)
            o.wfold.copy_(o.graph_out.detach())
            K.check(self.lib.savsr_pack_conv_chunks(self.ctx.handle, self.chunks_dev.data_ptr(), o.chunk_first, o.chunk_count, st))
        self._emit(fwd, launches=30, kind="island_osa")

    def _osa_backward(self, o: _Osa, producers: Sequence[int]) -> None:
        """After the per-sample weight gradients (dwfold) are in: backward of the fold island; the gradient of the pooled means
        joins the gradients of the producing convolutions through their grad_prep (cadd)."""
        def bwd(st):
            params = [self.P[n] for n in o.param_names]
            grads = torch.autograd.grad(o.graph_out, [o.leaf] + params, o.dwfold, allow_unused=True)
            o.dpool.copy_(grads[0])
            self._param_grads(o.param_names, grads[1:])
            o.dwfold.zero_()
            o.graph_out = None
        self._emit(bwd, launches=60, kind="island_osa")
        for s, slot in enumerate(producers):
            self.prep_mod.setdefault(slot, {})["cadd"] = (o.dpool.data_ptr() + s * 64 * 4, o.ci, 1.0 / float(self.npix))

    # ------------------------------------------------------------------ blocks
    def _osa_conv(self, prefixes: Sequence[str], srcs: Sequence[Sequence[int]], pools: Sequence[Sequence[torch.Tensor]], dsts: Sequence[int],
                  act: int) -> None:
        osas = [_Osa(self, p, srcs[d], pools[d]) for d, p in enumerate(prefixes)]
        self._keep.extend(osas)
        # builders run in reverse: the fold backward is registered FIRST so that it runs AFTER the conv backward (which produces dwfold)
        if self.native_attn:
            n = len(osas)
            pa = (K.OsaParams * n)(*[o.params for o in osas])
            ta = (K.OsaTrain * n)(*[o.extra for o in osas])
            ga = (K.OsaGrads * n)(*[o.grads for o in osas])
            self._keep += [pa, ta, ga]
            lib, ctx, B, npart, npix = self.lib, self.ctx.handle, self.B, self.npart, self.npix
            inv_h = float(np.float32(1.0) / np.float32(self.scale[0]))
            inv_w = float(np.float32(1.0) / np.float32(self.scale[1]))

            def bwd():
                self._emit(lambda st: K.check(lib.savsr_osa_fold_backward(ctx, pa, ta, ga, n, B, st)), launches=3, kind="osa_bwd")
                for d, o in enumerate(osas):
                    for s, slot in enumerate(srcs[d]):
                        self.prep_mod.setdefault(slot, {})["cadd"] = (o.dpool.data_ptr() + s * 64 * 4, o.ci, 1.0 / float(npix))
            self._builders.append(bwd)
            self._emit(lambda st: K.check(lib.savsr_osa_prologue_train(ctx, pa, ta, n, B, npart, npix, inv_h, inv_w, st)), launches=4, kind="osa_fwd")
        else:
            for d, o in enumerate(osas):
                self._builders.append(lambda o=o, d=d: self._osa_backward(o, srcs[d]))
            for o in osas:
                self._osa_fold(o)
        self._conv([_Spec(srcs[d], dsts[d], osa=osas[d], act=act) for d in range(len(prefixes))])

    def _residual_block(self, prefixes: Sequence[str], xs: Sequence[Sequence[int]]) -> List[List[int]]:
        """ResidualBlock.forward (savsr_arch.py:399-415) for len(prefixes) independent blocks per launch."""
        nd, nfr = len(prefixes), len(xs[0])
        use_os = (prefixes[0] + ".osconv.weight") in self.P
        new = self._new_slot
        tmp = [[new() for _ in range(nfr)] for _ in range(nd)]
        pools = [[self._buf(self.B, self.npart, 64) if use_os else None for _ in range(nfr)] for _ in range(nd)]
        self._conv([_Spec([xs[d][i]], tmp[d][i], f"{p}.conv0.{i}.weight", bias=f"{p}.conv0.{i}.bias", act=L_ACT, pool=pools[d][i])
                    for d, p in enumerate(prefixes) for i in range(nfr)])
        base = [new() for _ in range(nd)]
        if use_os:
            self._osa_conv([p + ".osconv" for p in prefixes], tmp, pools, base, L_ACT)
        else:
            self._conv([_Spec(tmp[d], base[d], p + ".conv1.weight", bias=p + ".conv1.bias", act=L_ACT, ksize=1) for d, p in enumerate(prefixes)], ksize=1)
        a = [[new() for _ in range(nfr)] for _ in range(nd)]
        self._conv([_Spec([base[d], tmp[d][i]], a[d][i], f"{p}.conv2.{i}.weight", bias=f"{p}.conv2.{i}.bias", act=L_ACT)
                    for d, p in enumerate(prefixes) for i in range(nfr)])
        outs = [[new() for _ in range(nfr)] for _ in range(nd)]
        self._add([(outs[d][i], xs[d][i], a[d][i]) for d in range(nd) for i in range(nfr)])
        return outs

    def _rcab(self, prefix: str, x: int) -> int:
        """RCAB (savsr_arch.py:504-549): conv-ReLU-conv, channel attention from the conv epilogue's pooled sums, x + t * y."""
        new = self._new_slot
        t1, t2, out = new(), new(), new()
        pool = self._buf(self.B, self.npart, 64)
        y = self._buf(self.B, 64)
        dy = self._buf(self.B, 64)
        dmean = self._buf(self.B, 64)
        self._conv([_Spec([x], t1, prefix + ".0.weight", bias=prefix + ".0.bias", act=K.ACT_RELU)])
        self._conv([_Spec([t1], t2, prefix + ".2.weight", bias=prefix + ".2.bias", pool=pool)])
        names = [prefix + ".3.attention.1.weight", prefix + ".3.attention.1.bias", prefix + ".3.attention.3.weight", prefix + ".3.attention.3.bias"]
        w1, b1, w2, b2 = (self.P[n] for n in names)
        lib, ctx, npart = self.lib, self.ctx.handle, self.npart
        self._emit(lambda st: K.check(lib.savsr_ca_scale_residual(ctx, self._ah(), t2, x, out, pool.data_ptr(), npart, w1.data_ptr(), b1.data_ptr(),
                                                                  w2.data_ptr(), b2.data_ptr(), y.data_ptr(), st)), launches=2, kind="ca")

        def bwd():
            if out not in self.gmap:
                return
            g = self.gmap[out]
            if self.native_attn:
                gp = [self.G[n] for n in names]
                npix = self.npix
                self._emit(lambda st: K.check(lib.savsr_slot_channel_dot(ctx, self._ah(), g, t2, dy.data_ptr(), st)), kind="ca_bwd")
                self._emit(lambda st: K.check(lib.savsr_ca_backward(ctx, pool.data_ptr(), npart, npix, self.B, w1.data_ptr(), b1.data_ptr(), w2.data_ptr(),
                                                                    b2.data_ptr(), y.data_ptr(), dy.data_ptr(), gp[0].data_ptr(), gp[1].data_ptr(),
                                                                    gp[2].data_ptr(), gp[3].data_ptr(), dmean.data_ptr(), st)), kind="ca_bwd")
            else:
                def run(st):
                    do = self._slot_view(g).float()
                    tt = self._slot_view(t2).float()
                    dy.copy_((do * tt).sum(dim=(1, 2)))
                    mean = (pool.sum(1) / float(self.npix)).detach().requires_grad_(True)
                    with torch.enable_grad():
                        yy = torch.sigmoid(F.linear(F.relu(F.linear(mean, w1.view(w1.shape[0], -1), b1)), w2.view(w2.shape[0], -1), b2))
                    grads = torch.autograd.grad(yy, [mean, w1, b1, w2, b2], dy)
                    dmean.copy_(grads[0])
                    self._param_grads(names, grads[1:])
                self._emit(run, launches=25, kind="island_ca")
            self.gmap[t2] = g
            self.shared.add(g)
            self.prep_mod[t2] = {"cscale": (y.data_ptr(), 64), "cadd": (dmean.data_ptr(), 64, 1.0 / float(self.npix))}
            self._accumulate([(x, g)])
        self._builders.append(bwd)
        return out

    def _slot_view(self, slot: int) -> torch.Tensor:
        return self.arena_t[slot * self.B:(slot + 1) * self.B]

    def _osadapt(self, prefix: str, r_slot: int, plr: torch.Tensor, share: int) -> int:
        """OSAdapt (savsr_arch.py:186-214) + `+ gamma * share` (727-732): the OSA-Conv is native, the mask net and the combination
        h = R + adapted * mask(R) + gamma * share run as an ATen island."""
        a = self._new_slot()
        out = self._new_slot()
        self._osa_conv([prefix + ".adapt"], [[r_slot]], [[plr]], [a], K.ACT_NONE)
        if self.native_mask:
            self._osadapt_native(prefix, r_slot, a, share, out)
            return out
        net = self.net
        m = prefix + ".mask"
        names = [f"{m}.{i}.{k}" for i in (0, 1, 4, 5, 7, 8, 11, 12) for k in ("weight", "bias")] + ["gamma"]
        st8 = {}

        def fwd(st):
            leaves = [self._export(s).requires_grad_(True) for s in (r_slot, a, share)]
            with torch.enable_grad():
                hh = leaves[0] + leaves[1] * T.osadapt_mask(net, prefix, leaves[0]) + self.P["gamma"] * leaves[2]
            st8["leaves"], st8["out"] = leaves, hh
            self._import(out, hh.detach())
        self._emit(fwd, launches=40, kind="island_osadapt")

        def bwd():
            if out not in self.gmap:
                return
            g = self.gmap[out]

            def run(st):
                dh = self._export(g)
                params = [self.P[n] for n in names]
                grads = torch.autograd.grad(st8["out"], st8["leaves"] + params, dh, allow_unused=True)
                st8["grads"] = grads[:3]
                self._param_grads(names, grads[3:])
                st8["out"] = None
            self._emit(run, launches=80, kind="island_osadapt")
            self._import_grads([(s, (lambda i=i: st8["grads"][i])) for i, s in enumerate((r_slot, a, share))])
        self._builders.append(bwd)
        return out

    def _osadapt_native(self, prefix: str, r_slot: int, a: int, share: int, out: int) -> None:
        """Mask net + combination on the native kernels (train_mask.cu): the 64 -> 16 convolution forward / dgrad / wgrad on tensor cores
        (N = 16 forward; its gradient as a 16-of-64-channel arena slot through the ordinary data- / weight-gradient path), the rest on
        CUDA cores with batch-statistics BatchNorm."""
        B, P, Q, dev = self.B, self.npix, (self.h // 2) * (self.w // 2), self.device
        Pm, G, Bf = self.P, self.G, self.net.B
        lib, ctx = self.lib, self.ctx.handle
        m = prefix + ".mask"
        if self._mask_scratch is None:             # backward scratch shared by the four OSAdapts of the plan (they run one after the other)
            z = lambda *sh, dt=torch.float32: self._buf(*sh, dtype=dt)      # noqa: E731
            self._mask_scratch = dict(dmask=z(B, P), dm11=z(B, P), dt4=z(B, Q, 16), dm7=z(B, Q, 16), dt3=z(B, Q, 16), dm4=z(B, Q, 16), dt2=z(B, Q, 16),
                                      sums=z(64, dt=torch.float64), dm0_slot=self._new_slot())
        sc = self._mask_scratch
        act = dict(m0=self._buf(B, P, 16), t2=self._buf(B, Q, 16), m4=self._buf(B, Q, 16), t3=self._buf(B, Q, 16), m7=self._buf(B, Q, 16),
                   t5=self._buf(B, P, 16), m11=self._buf(B, P), mask=self._buf(B, P), stat=self._buf(4 * 32), coef=self._buf(4 * 48))
        mt = K.MaskTrain()
        mt.w4, mt.b4, mt.w7, mt.b7 = (Pm[f"{m}.{k}"].data_ptr() for k in ("4.weight", "4.bias", "7.weight", "7.bias"))
        mt.w11, mt.b11 = Pm[m + ".11.weight"].data_ptr(), Pm[m + ".11.bias"].data_ptr()
        mt.d_w4, mt.d_b4, mt.d_w7, mt.d_b7 = (G[f"{m}.{k}"].data_ptr() for k in ("4.weight", "4.bias", "7.weight", "7.bias"))
        mt.d_w11, mt.d_b11 = G[m + ".11.weight"].data_ptr(), G[m + ".11.bias"].data_ptr()
        for l, idx in enumerate((1, 5, 8, 12)):
            mt.bn_w[l], mt.bn_b[l] = Pm[f"{m}.{idx}.weight"].data_ptr(), Pm[f"{m}.{idx}.bias"].data_ptr()
            mt.d_bn_w[l], mt.d_bn_b[l] = G[f"{m}.{idx}.weight"].data_ptr(), G[f"{m}.{idx}.bias"].data_ptr()
            mt.bn_rm[l], mt.bn_rv[l] = Bf[f"{m}.{idx}.running_mean"].data_ptr(), Bf[f"{m}.{idx}.running_var"].data_ptr()
            nbt = f"{m}.{idx}.num_batches_tracked"
            if nbt in Bf:
                self.nbt_counts[nbt] = self.nbt_counts.get(nbt, 0) + 1
        mt.gamma, mt.d_gamma = Pm["gamma"].data_ptr(), G["gamma"].data_ptr()
        mt.momentum, mt.eps = T.BN_MOMENTUM, T.BN_EPS
        for k, v in act.items():
            setattr(mt, k, v.data_ptr())
        for k in ("dmask", "dm11", "dt4", "dm7", "dt3", "dm4", "dt2", "sums"):
            setattr(mt, k, sc[k].data_ptr())
        self._keep.append(mt)
        # forward: pack the 64 -> 16 filter (N = 16 blocks), convolve into m0, then the rest of the net
        w0, b0 = Pm[m + ".0.weight"], Pm[m + ".0.bias"]
        packed16 = self._buf(int(lib.savsr_packed_weight_bytes(16, 64, 3)), dtype=torch.uint8)
        self._emit(lambda st: K.check(lib.savsr_pack_conv_weight(w0.data_ptr(), 16, 16, 64, 3, 16, self.fmt, K.ROWS_LINEAR, packed16.data_ptr(), st)), kind="mask_fwd")
        g0 = self._group([r_slot], 0, packed16.data_ptr(), b0.data_ptr())
        g0.aux_dst = act["m0"].data_ptr()
        arr = (K.ConvGroup * 1)(g0)
        self._keep.append(arr)
        self._emit(lambda st: K.check(lib.savsr_conv(ctx, self._ah(), arr, 1, 3, 16, K.DST_AUX16, K.IMPL_HALO, st)), kind="mask_fwd")
        self._emit(lambda st: K.check(lib.savsr_mask_forward_train(ctx, self._ah(), C.byref(mt), r_slot, a, share, out, st)), launches=14, kind="mask_fwd")
        wkey = m + ".0.weight"

        def bwd():
            if out not in self.gmap:
                return
            g = self.gmap[out]
            da, gs, dm0 = self._new_slot(), self._new_slot(), sc["dm0_slot"]
            self._emit(lambda st: K.check(lib.savsr_mask_backward_train(ctx, self._ah(), C.byref(mt), g, a, share, da, gs, dm0, st)), launches=22, kind="mask_bwd")
            self.gmap[a] = da                                      # a has one consumer: this is its whole gradient
            self._accumulate([(r_slot, g), (share, gs)])
            # the 64 -> 16 convolution: its output gradient sits in channels 0..15 of slot dm0 (the rest zero)
            gt = self._new_tslots(1)
            dw64 = self.W.scratch_grad(("mask0.w", prefix), (64, 64, 3, 3), scatter_to=G[wkey], rows=16)
            db64 = self.W.scratch_grad(("mask0.b", prefix), (64,), scatter_to=G[m + ".0.bias"], rows=16)
            e = K.GradPrep()
            e.dv_slot, e.out_slot, e.g_slot, e.gt_tslot, e.act, e.slope = dm0, -1, -1, gt, K.ACT_NONE, 0.0
            e.cscale, e.cscale_stride, e.cadd, e.cadd_stride, e.cadd_mul = None, 0, None, 0, 0.0
            e.dbias = db64.data_ptr()
            parr = (K.GradPrep * 1)(e)
            self._keep.append(parr)
            self._emit(lambda st: K.check(lib.savsr_grad_prep(ctx, self._ah(), self.tarena.data_ptr(), self.n_tslots, self.pitch, parr, 1, st)), kind="grad_prep")
            d, r = self._gdst(r_slot)
            self._conv_launch([self._group([dm0], d, self.W.dgrad(((wkey, 0, 0),)), res1=r, src_channels=16)])
            it = K.WgradItem()
            it.g_tslot, it.ksize, it.dw, it.ci_total, it.ci_off, it.o_off = gt, 3, dw64.data_ptr(), 64, 0, 0
            it.per_sample, it.sample_stride, it.layout = 0, 0, K.WGRAD_OIHW
            self._wsrc.append(r_slot)
            self.witems.append(it)
            self.deferred.append(len(self.witems) - 1)
        self._builders.append(bwd)

    # ------------------------------------------------------------------ program construction
    def _build(self) -> None:
        B, t = self.B, 7
        lib, ctx = self.lib, self.ctx.handle
        new = self._new_slot
        self._wsrc: List[int] = []
        self._keep_step: List[torch.Tensor] = []
        tiles = ((self.w + K.TILE_W - 1) // K.TILE_W) * ((self.h + K.TILE_H - 1) // K.TILE_H)
        self.npart = tiles * 4
        ZERO, FR = new(), new()
        self.noreq = {ZERO, FR}
        self.x_in = self._buf(B, t, 3, self.h, self.w)
        self.gt = self._buf(B, 3, self.H, self.Wd)
        xin, hh, ww = self.x_in.data_ptr(), self.h, self.w
        self._emit(lambda st: K.check(lib.savsr_pack_frames(ctx, self._ah(), xin, t, hh, ww, FR, st)), kind="pack_frames")
        dirs = ("f2p_win", "p2f_win")
        n_it = t - 3 + 1
        Fs: List[List[int]] = [[0] * n_it for _ in dirs]
        hpast = [ZERO, ZERO]
        for idx in range(n_it):
            centre = [t - 2 - idx, idx + 1]
            s0 = [[new(), new()] for _ in dirs]
            specs = []
            for d, p in enumerate(dirs):
                c = centre[d]
                specs.append(_Spec([FR], s0[d][0], self.W.expand_first_layer(p, "conv_c", c), bias=p + ".conv_c.bias", act=L_ACT, src_channels=32))
                specs.append(_Spec([FR], s0[d][1], self.W.expand_first_layer(p, "conv_sup", c), bias=p + ".conv_sup.bias", act=L_ACT, src_channels=32))
            self._conv(specs)
            cur = [[s0[d][0], s0[d][1], hpast[d]] for d in range(2)]
            for j in range(4):
                cur = self._residual_block([f"{p}.blocks.{j}" for p in dirs], cur)
            fd = [new(), new()]
            self._conv([_Spec(cur[d], fd[d], p + ".merge.weight", bias=p + ".merge.bias") for d, p in enumerate(dirs)])
            hpast = fd
            for d in range(2):
                Fs[d][idx] = fd[d]
        # pyramid fusion, WindowUnit_l2 (savsr_arch.py:485-501, 721-723)
        p2 = "h_win.0"
        gx = [new() for _ in range(5)]
        self._conv([_Spec([Fs[0][n_it - 1 - i], Fs[1][i]], gx[i], f"{p2}.conv_h.{i}.weight", bias=f"{p2}.conv_h.{i}.bias", act=L_ACT) for i in range(5)])
        cur5 = gx
        for j in range(2):
            cur5 = self._residual_block([f"{p2}.blocks.{j}"], [cur5])[0]
        M = [new(), new()]
        self._conv([_Spec(cur5, M[k], p2 + ".merge.weight", half=k, bias=p2 + ".merge.bias") for k in range(2)])
        A = new()
        self._conv([_Spec(M, A, "h_win_conv_h.weight", bias="h_win_conv_h.bias", act=L_ACT)])
        # reconstruction: 4 x (ResidualGroup -> OSAdapt -> + gamma * share) (savsr_arch.py:727-734)
        h_cur = A
        for gi in range(4):
            x = h_cur
            for r in range(8):
                x = self._rcab(f"RG.{gi}.residual_group.{r}.rcab", x)
            R = new()
            plr = self._buf(B, self.npart, 64)
            self._conv([_Spec([x], R, f"RG.{gi}.conv.weight", bias=f"RG.{gi}.conv.bias", res1=h_cur, pool=plr)])
            h_cur = self._osadapt(f"adapt.{gi}", R, plr, A)
        TR = new()
        self._conv([_Spec([h_cur], TR, "conv_last.weight", bias="conv_last.bias", res1=A)])
        # SATU + tail + bilinear skip + Charbonnier: ATen island (savsr_arch.py:315-376, 738-739; basic_loss.py:22-24)
        net = self.net
        st8: dict = {}
        names = [n for n in self.P if n.startswith("upsample.") or n.startswith("tail.")]

        def satu_fwd(st):
            leaves = [self._export(s).requires_grad_(True) for s in (TR, A)]
            tf32 = torch.backends.cuda.matmul.allow_tf32
            torch.backends.cuda.matmul.allow_tf32 = True        # the expert mixes and their weight gradients (K = B*H*W) on tensor cores, like the convs around them
            try:
                with torch.enable_grad():
                    sr = net.conv("tail", T.satu(net, "upsample", leaves[0], self.scale, leaves[1]))
                    sr = sr + F.interpolate(self.x_in[:, t // 2], size=(self.H, self.Wd), mode="bilinear", align_corners=False)
                    loss = T.charbonnier(sr, self.gt) if self.own_loss else None
            finally:
                torch.backends.cuda.matmul.allow_tf32 = tf32
            self.sr = sr.detach()
            self.loss = loss.detach() if loss is not None else None
            st8["leaves"], st8["sr"], st8["loss"] = leaves, sr, loss

        def satu_bwd(st):
            params = [self.P[n] for n in names]
            tf32 = torch.backends.cuda.matmul.allow_tf32
            torch.backends.cuda.matmul.allow_tf32 = True
            try:
                if self.own_loss:
                    grads = torch.autograd.grad(st8["loss"], st8["leaves"] + params, allow_unused=True)
                else:                                           # the caller's loss: its gradient w.r.t. the output arrives in self.dsr
                    grads = torch.autograd.grad(st8["sr"], st8["leaves"] + params, self.dsr, allow_unused=True)
            finally:
                torch.backends.cuda.matmul.allow_tf32 = tf32
            st8["grads"] = grads[:2]
            self._param_grads(names, grads[2:])
            st8["sr"] = st8["loss"] = None
        self._emit(satu_fwd, launches=150, kind="island_satu")
        self._satu_bwd = satu_bwd
        self.kinds[id(satu_bwd)] = "bwd:island_satu"

        # ---- backward program: builders in reverse order of the forward
        self._emit_to = self.bwd_ops
        self._emit(self._satu_bwd, launches=250, kind="island_satu")
        self._import_grads([(s, (lambda i=i: st8["grads"][i])) for i, s in enumerate((TR, A))])
        # ops up to the last import read tensors autograd produced this step (eager); everything after works on fixed buffers
        self.n_bwd_island = 1 + max(i for i, op in enumerate(self.bwd_ops) if self.kinds.get(id(op)) == "bwd:import")
        for b in reversed(self._builders):
            b()
        # every weight gradient that was deferred, in one persistent launch
        if self.deferred:
            order = self.deferred
            self._x3([self._wsrc[i] for i in order])
        # ---- allocate, now that slot counts are known
        # The arenas depend on (batch, h, w) and on the op list, not on the scale: every plan of one configuration has the SAME slot
        # layout (the build is deterministic), plans run one after the other, and every slot is rewritten by each step -- so all
        # scales share one pair of arenas (5.5 GB at 4 x 64 x 64) instead of owning one each (the training YAML rotates 60 scales).
        akey = ("arenas", B, self.h, self.w, self.native_attn, self.native_mask, self.n_slots, self.n_tslots)
        shared = self.W._bufs.get(akey)
        if shared is None:
            shared = self.W._bufs[akey] = (
                torch.zeros(self.n_slots * B, self.h, self.w, 64, dtype=torch.bfloat16, device=self.device),
                torch.zeros(max(self.n_tslots, 1) * B * 64 * self.h * self.pitch, dtype=torch.bfloat16, device=self.device))
        self.arena_t, self.tarena = shared
        self.arena = K.Arena(self.ctx, self.arena_t.data_ptr(), self.n_slots, B, self.h, self.w)
        # weight-gradient table: inline (OSA) items keep their indices, the deferred ones are gathered behind them
        items = list(self.witems)
        for i, it in enumerate(items):
            it.x_tslot = self.x3_of[self._wsrc[i]]
        table = items + [items[i] for i in self.deferred]
        d_first, d_count = len(items), len(self.deferred)
        arr = (K.WgradItem * len(table))(*table)
        self.witems_dev = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).to(self.device)
        if d_count:
            self._wgrad_launch(d_first, d_count)
        carr = (K.PackChunk * max(len(self.chunks), 1))(*self.chunks)
        self.chunks_dev = torch.frombuffer(bytearray(bytes(carr)), dtype=torch.uint8).to(self.device)
        self._emit_to = self.fwd_ops
        self.nbytes = self.arena_t.numel() * 2 + self.tarena.numel() * 2

    # ------------------------------------------------------------------ execution
    def run_forward_native(self, join: bool) -> None:
        """Every forward op except the SATU island, plus (on a side stream) the x-shifted NCHW copies the weight gradient needs."""
        with torch.cuda.device(self.device), pdl(self.ctx, True):
            self.ctx.set_format(self.fmt)
            main = torch.cuda.current_stream(self.device)
            st = main.cuda_stream
            for op in self.fwd_ops[:-1]:
                op(st)
            if self._side is None:
                self._side = torch.cuda.Stream(self.device)
            self._side.wait_stream(main)                      # fork: the transposed copies of the activations (weight-gradient operands)
            with torch.cuda.stream(self._side):
                sst = self._side.cuda_stream
                for op in self.x3_ops:
                    op(sst)
            if join:
                main.wait_stream(self._side)

    def run_forward_island(self) -> None:
        """SATU's HR side + tail (+ loss): the ATen island, and the BatchNorm call counters."""
        with torch.cuda.device(self.device):
            self._keep_step.clear()
            self.fwd_ops[-1](torch.cuda.current_stream(self.device).cuda_stream)
            if self.nbt_counts:                               # BatchNorms evaluated by native kernels: one counter bump per forward call, as nn.BatchNorm2d does
                torch._foreach_add_([self.net.B[n] for n in self.nbt_counts], [int(c) for c in self.nbt_counts.values()])

    def run_forward(self) -> None:
        """Forward of the launch list on the device's current stream (x_in -> sr, and the loss against self.gt when the plan owns it)."""
        self.run_forward_native(join=False)
        self.run_forward_island()                             # ... overlaps the side stream's copies
        with torch.cuda.device(self.device):
            torch.cuda.current_stream(self.device).wait_stream(self._side)      # join

    def run_backward_island(self, dsr: Optional[torch.Tensor] = None) -> None:
        """Backward of the SATU island (autograd) and the import of its input gradients into arena slots."""
        with torch.cuda.device(self.device), pdl(self.ctx, True):
            self.ctx.set_format(self.fmt)
            st = torch.cuda.current_stream(self.device).cuda_stream
            self.dsr = dsr
            for op in self.bwd_ops[:self.n_bwd_island]:
                op(st)
            self.dsr = None

    def run_backward_native(self) -> None:
        """Every other backward op: pure launches on fixed buffers (graph-capturable without any autograd inside)."""
        with torch.cuda.device(self.device), pdl(self.ctx, True):
            self.ctx.set_format(self.fmt)
            st = torch.cuda.current_stream(self.device).cuda_stream
            for op in self.bwd_ops[self.n_bwd_island:]:
                op(st)

    def run_backward(self, dsr: Optional[torch.Tensor] = None) -> None:
        """Backward of the launch list; gradients are ACCUMULATED into the flat gradient buffer.  dsr: gradient of the caller's loss
        w.r.t. the output (plans built with own_loss=False)."""
        self.run_backward_island(dsr)
        self.run_backward_native()

    def run(self, x: Optional[torch.Tensor] = None, gt: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Forward + loss + backward on the device's current stream; gradients are ACCUMULATED into the flat gradient buffer
        (the caller zeroes it and has packed the weights: NativeTrainer does both).  Returns the loss (device scalar)."""
        with torch.cuda.device(self.device):
            if x is not None:
                self.x_in.copy_(x, non_blocking=True)
            if gt is not None:
                self.gt.copy_(gt, non_blocking=True)
        self.run_forward()
        self.run_backward()
        return self.loss

    def run_profiled(self) -> Dict[str, Dict[str, float]]:
        """Eager forward + backward with a CUDA-event pair around every op: {phase:kind: {"ms", "ops"}} (islands include their ATen launches)."""
        out: Dict[str, Dict[str, float]] = {}
        with torch.cuda.device(self.device):
            self.ctx.set_format(self.fmt)
            stream = torch.cuda.current_stream(self.device)
            st = stream.cuda_stream
            self._keep_step.clear()
            evs = []
            for op in self.fwd_ops + self.x3_ops + self.bwd_ops:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                op(st)
                e1.record(stream)
                evs.append((self.kinds.get(id(op), "?"), e0, e1))
            stream.synchronize()
        for kind, e0, e1 in evs:
            d = out.setdefault(kind, dict(ms=0.0, ops=0))
            d["ms"] += e0.elapsed_time(e1); d["ops"] += 1
        return out


# ====================================================================================================== trainer
class NativeTrainer:
    """The optimisation step of lbasicsr/models/sr_model.py:101-128 on the native plan: pack weights -> forward -> Charbonnier ->
    backward -> (all-reduce of the flat gradient over NCCL when torch.distributed is initialised) -> Adam + EMA, one CUDA graph per
    (scale, batch shape).  lr / betas: the train YAML's Adam (2e-4, 0.9 / 0.99); EMA 0.999 (base_model.py:75-82).
    `optimizer` (FlatAdam) takes the caller's lr schedulers and checkpoints in torch.optim.Adam's layout; ema_state_dict() is the EMA
    network's full state_dict (params_ema); training_state() / resume() are BasicSR's .state file."""

    def __init__(self, net: torch.nn.Module, lr: float = 2e-4, betas=(0.9, 0.99), eps: float = 1e-8, ema_decay: float = 0.999,
                 use_graph: bool = True, world_size: int = 1, native_attn: bool = True, native_mask: bool = True):
        self.net = net
        self.native_attn, self.native_mask = native_attn, native_mask
        self.flat = FlatParams(net, ema=ema_decay > 0)
        dev = self.flat.device
        self.ctx = context(_dev_index(dev))
        self.weights = TrainWeights(self.flat, self.ctx)
        self.ema_decay = ema_decay
        self.world = world_size
        self.optimizer = FlatAdam(self.flat, self.ctx, lr=lr, betas=betas, eps=eps, ema_decay=ema_decay, world_size=world_size, use_graph=use_graph)
        self.use_graph = use_graph
        self.plans: Dict[tuple, TrainPlan] = {}
        self._graphs: Dict[int, tuple] = {}
        self._ema_buffers = self._snapshot_buffers(net.state_dict())

    # ---- hyper-parameters: the optimizer's group, which schedulers rewrite
    @property
    def lr(self) -> float:
        return self.optimizer.param_groups[0]["lr"]

    @lr.setter
    def lr(self, value: float) -> None:
        self.optimizer.param_groups[0]["lr"] = value

    @property
    def betas(self) -> tuple:
        return tuple(self.optimizer.param_groups[0]["betas"])

    @property
    def eps(self) -> float:
        return self.optimizer.param_groups[0]["eps"]

    @property
    def use_graph(self) -> bool:
        return self._use_graph

    @use_graph.setter
    def use_graph(self, value: bool) -> None:
        self._use_graph = self.optimizer.use_graph = bool(value)

    # ---- EMA in the reference's layout
    @property
    def ema(self) -> Optional[Dict[str, torch.Tensor]]:
        return {n: self.flat.ema_view(n) for n in self.flat.P} if self.flat.ema is not None else None

    def _snapshot_buffers(self, sd: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        """BasicSR's model_ema averages named_parameters() only: net_g_ema keeps the buffers (BatchNorm running statistics, call
        counters) it was built or loaded with.  So do we: a copy of the buffers taken when the EMA is initialised."""
        return {k: v.detach().clone() for k, v in sd.items() if k not in self.flat.P}

    def ema_state_dict(self) -> Optional[Dict[str, torch.Tensor]]:
        """The EMA network's full state_dict (every key of net.state_dict(), in its order), the `params_ema` of a BasicSR checkpoint:
        the averaged parameters (views of the flat EMA buffer) and the buffers snapshot at construction / load_ema_state_dict.
        None when the trainer keeps no EMA (ema_decay 0)."""
        if self.flat.ema is None:
            return None
        return {k: (self.flat.ema_view(k) if k in self.flat.P else self._ema_buffers[k]) for k in self.net.state_dict()}

    def load_ema_state_dict(self, sd: Dict[str, torch.Tensor]) -> None:
        """Reverse of ema_state_dict, with strict key checking: parameters into the flat EMA buffer, buffers into the snapshot."""
        if self.flat.ema is None:
            raise ValueError("this trainer keeps no EMA (ema_decay 0)")
        want = self.net.state_dict()
        missing, unexpected = [k for k in want if k not in sd], [k for k in sd if k not in want]
        if missing or unexpected:
            raise ValueError(f"EMA state_dict keys differ from the network's: missing {missing[:4]} ({len(missing)}), "
                             f"unexpected {unexpected[:4]} ({len(unexpected)})")
        for k, v in want.items():
            if tuple(sd[k].shape) != tuple(v.shape):
                raise ValueError(f"EMA state_dict: {k} has shape {tuple(sd[k].shape)}, the network {tuple(v.shape)}")
        with torch.no_grad():
            for n in self.flat.P:
                self.flat.ema_view(n).copy_(sd[n])
        self._ema_buffers = {k: sd[k].detach().to(want[k].device, want[k].dtype, copy=True) for k in want if k not in self.flat.P}

    # ---- BasicSR's training state (base_model.py save_training_state / resume_training)
    def training_state(self, iter: int, epoch: int, schedulers: Sequence = ()) -> dict:
        """{'epoch', 'iter', 'optimizers': [optimizer state], 'schedulers': [their states]}: the .state file BasicSR writes."""
        return {"epoch": epoch, "iter": iter, "optimizers": [self.optimizer.state_dict()], "schedulers": [s.state_dict() for s in schedulers]}

    def resume(self, state: dict, schedulers: Sequence = ()) -> Tuple[int, int]:
        """Load a training_state() (or BasicSR's resume state for one Adam) into the optimizer and `schedulers`; returns (epoch, iter).
        With several ranks every rank loads the same state."""
        opts, scheds = state["optimizers"], state["schedulers"]
        if len(opts) != 1:
            raise ValueError(f"the state holds {len(opts)} optimizers; NativeTrainer has one")
        if len(scheds) != len(schedulers):
            raise ValueError(f"the state holds {len(scheds)} schedulers, {len(schedulers)} were given")
        self.optimizer.load_state_dict(opts[0])
        for s, sd in zip(schedulers, scheds):
            s.load_state_dict(sd)
        return state["epoch"], state["iter"]

    def plan_for(self, lq: torch.Tensor, scale) -> TrainPlan:
        b, t, c, h, w = lq.shape
        key = (tuple(normalize_scale(scale)), b, h, w)
        if key not in self.plans:
            self.plans[key] = TrainPlan(self.net, self.flat, self.weights, b, h, w, scale, native_attn=self.native_attn, native_mask=self.native_mask)
        return self.plans[key]

    def _fwd_bwd(self, plan: TrainPlan) -> torch.Tensor:
        st = torch.cuda.current_stream(self.flat.device).cuda_stream
        self.flat.g.zero_()
        self.weights.zero_scratch()
        self.weights.pack(st)
        loss = plan.run()
        self.weights.scatter_expanded_grads()
        return loss

    def _allreduce(self) -> None:
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(self.flat.g)          # one NCCL all-reduce of the flat gradient buffer (75.6 MB), summed; Adam divides

    def step(self, lq: torch.Tensor, gt: torch.Tensor, scale) -> torch.Tensor:
        """One optimisation step; returns the loss of this rank's batch (device scalar)."""
        self.net.set_scale(scale)
        self.net.train()
        plan = self.plan_for(lq, scale)
        dev = self.flat.device
        with torch.cuda.device(dev):
            plan.x_in.copy_(lq, non_blocking=True)
            plan.gt.copy_(gt, non_blocking=True)
            if not self.use_graph:
                loss = self._fwd_bwd(plan)
                self._allreduce()
                self.optimizer.step()
                return loss
            key = id(plan)
            ent = self._graphs.get(key)
            if ent is None:
                # warm-up outside the graph (kernel attributes, allocator pools), with the BatchNorm statistics rolled back afterwards;
                # the optimizer is not run, so the weights are untouched
                bufs = [(b, b.clone()) for _, b in self.net.named_buffers()]
                side = torch.cuda.Stream(dev)
                side.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(side):
                    self._fwd_bwd(plan)
                torch.cuda.current_stream(dev).wait_stream(side)
                for b, saved in bufs:
                    b.copy_(saved)
                torch.cuda.synchronize(dev)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=torch.cuda.Stream(dev)):
                    loss = self._fwd_bwd(plan)
                ent = self._graphs[key] = (g, loss)
            g, loss = ent
            g.replay()
            self._allreduce()
            self.optimizer.step()                             # replays the optimizer's own graph (captured at its first step)
            return loss


# ====================================================================================================== the module's train-mode forward
class ModuleTraining:
    """What `SAVSR.forward` needs to run natively in train mode under SOMEBODY ELSE'S training loop -- the reference's
    `optimize_parameters` (lbasicsr/models/sr_model.py:101-128: net_g(lq), its own loss, backward(), its own torch.optim.Adam, model_ema),
    with or without DistributedDataParallel: flat parameter views, the packed weights, one plan per (scale, shape) built with
    own_loss=False.  The forward returns the output as an autograd node whose backward runs the plan's backward launch list.
    Both halves are replayed as CUDA graphs (captured on their second use, sharing one memory pool: the backward reads what the
    forward saved), so the ~1 400 launches of a step cost no host time."""

    def __init__(self, net: torch.nn.Module, native_attn: bool = True, native_mask: bool = True, use_graph: bool = True):
        self.net = net
        self.flat = FlatParams(net, ema=False, assign_grads=False)
        self.ctx = context(_dev_index(self.flat.device))
        self.weights = TrainWeights(self.flat, self.ctx)
        self.native_attn, self.native_mask = native_attn, native_mask
        self.use_graph = use_graph and native_attn and native_mask      # graphs hold native launches only: no ATen island may sit inside the trunk
        self.plans: Dict[tuple, TrainPlan] = {}
        self.params = list(self.flat.P.values())
        self.slices = [(self.flat.offsets[n], p.numel(), p.shape) for n, p in self.flat.P.items()]

    def plan_for(self, x: torch.Tensor, scale) -> TrainPlan:
        b, t, c, h, w = x.shape
        key = (tuple(normalize_scale(scale)), b, h, w)
        if key not in self.plans:
            plan = TrainPlan(self.net, self.flat, self.weights, b, h, w, scale, native_attn=self.native_attn, native_mask=self.native_mask, own_loss=False)
            plan.dsr_buf = torch.zeros(b, 3, plan.H, plan.Wd, device=self.flat.device)
            plan.uses, plan.g_fwd, plan.g_bwd = 0, None, None
            self.plans[key] = plan
        return self.plans[key]

    @staticmethod
    def supports(x: torch.Tensor) -> bool:
        return (x.is_cuda and x.dim() == 5 and x.shape[1] == 7 and x.shape[3] % 2 == 0 and x.shape[4] % 2 == 0
                and x.shape[0] <= MAX_NATIVE_BATCH)

    def forward(self, x: torch.Tensor, scale) -> torch.Tensor:
        return _NativeNet.apply(x, self, self.plan_for(x, scale), *self.params)

    # ---- CUDA graphs hold the native launches only (no autograd inside a capture); the SATU island runs eagerly on both sides
    def _fwd_native(self, plan: TrainPlan) -> None:
        self.weights.pack(torch.cuda.current_stream(plan.device).cuda_stream)      # the caller's optimizer changed the weights since the last step
        plan.run_forward_native(join=True)

    def _bwd_native(self, plan: TrainPlan) -> None:
        plan.run_backward_native()
        self.weights.scatter_expanded_grads()

    def run_forward(self, plan: TrainPlan) -> None:
        dev = plan.device
        plan.uses += 1
        if not self.use_graph or plan.uses == 1 or torch.cuda.is_current_stream_capturing():     # (inside somebody else's capture: just record)
            self._fwd_native(plan)
        elif plan.g_fwd is None:
            # second use: capture BOTH graphs here, on the caller's thread (the backward itself runs on autograd's worker thread)
            torch.cuda.synchronize(dev)
            cap = torch.cuda.Stream(dev)
            gf = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gf, stream=cap):
                self._fwd_native(plan)
            gb = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gb, stream=cap):
                self._bwd_native(plan)
            plan.g_fwd, plan.g_bwd = gf, gb
            gf.replay()                                  # capture does not execute
        else:
            plan.g_fwd.replay()
        plan.run_forward_island()

    def run_backward(self, plan: TrainPlan) -> None:
        self.flat.g.zero_()
        self.weights.zero_scratch()
        plan.run_backward_island(plan.dsr_buf)
        if plan.g_bwd is not None and not torch.cuda.is_current_stream_capturing():
            plan.g_bwd.replay()
        else:
            self._bwd_native(plan)


class _NativeNet(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x: torch.Tensor, state: ModuleTraining, plan: TrainPlan, *params):
        with torch.cuda.device(plan.device):
            plan.x_in.copy_(x.detach(), non_blocking=True)
            state.run_forward(plan)
            out = plan.sr.clone()
        ctx.state, ctx.plan = state, plan
        return out

    @staticmethod
    def backward(ctx, dsr: torch.Tensor):
        state, plan = ctx.state, ctx.plan
        with torch.cuda.device(plan.device):
            plan.dsr_buf.copy_(dsr.detach(), non_blocking=True)
            state.run_backward(plan)
            g = state.flat.g.clone()                  # autograd may keep what we return as p.grad: hand out a private copy, not views of the scratch
        return (None, None, None) + tuple(g[o:o + k].view(shape) for o, k, shape in state.slices)
