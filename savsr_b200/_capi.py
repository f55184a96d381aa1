"""ctypes binding of libsavsr_sm100.so (include/savsr_b200.h).

This is the reference-side FFI stub a maintainer of the (pure-Python) reference would add: plain
pointers, sizes and a stream, nothing torch-specific crosses the boundary.  There is NO fallback:
if the shared library is missing or a call fails, a Python exception is raised, mirroring the
reference's convention of raising from its native ops (ops/dcn/src/deform_conv_ext.cpp:64-67).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

ABI_VERSION = 4
MAX_SRC = 5
MAX_GROUPS = 25
TILE_W, TILE_H = 8, 16

ACT_NONE, ACT_LRELU, ACT_RELU = 0, 1, 2
DST_ARENA, DST_AUX16 = 0, 1
IMPL_TAP, IMPL_HALO, IMPL_CHECK = 0, 1, 2
IMPL_NAMES = {"tap": IMPL_TAP, "halo": IMPL_HALO, "check": IMPL_CHECK}
FMT_BF16, FMT_FP16 = 0, 1
FMT_NAMES = {"bf16": FMT_BF16, "fp16": FMT_FP16}
OPT_BIGK_ALL, OPT_BIGK_ISSUERS, OPT_PDL = 0, 1, 2   # enum savsr_option
WGRAD_OIHW, WGRAD_TIO = 0, 1     # enum savsr_wgrad_layout
ROWS_LINEAR, ROWS_QUAD = 0, 1     # enum savsr_row_order: QUAD for everything savsr_conv / savsr_satu_kconv_sta consume with n_tile 64
SCENE_SCRATCH_WORDS = 1024        # SAVSR_SCENE_SCRATCH_WORDS: uint64 scratch of one scene detector

# SAVSR_LIB_PATH: alternative build of the same ABI (A/B timing of kernel variants); default = the in-tree library
LIB_PATH = os.environ.get("SAVSR_LIB_PATH") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libsavsr_sm100.so")


class SavsrError(RuntimeError):
    """A libsavsr_sm100 call returned non-zero."""


class ConvGroup(C.Structure):
    _fields_ = [
        ("src_slot", C.c_int32 * MAX_SRC),
        ("nsrc", C.c_int32),
        ("dst_slot", C.c_int32),
        ("res1_slot", C.c_int32),
        ("res2_slot", C.c_int32),
        ("res2_scale", C.c_float),
        ("act", C.c_int32),
        ("slope", C.c_float),
        ("weight", C.c_void_p),
        ("weight_sample_stride", C.c_int64),
        ("bias", C.c_void_p),
        ("mask", C.c_void_p),
        ("pool", C.c_void_p),
        ("aux_dst", C.c_void_p),
        ("src_channels", C.c_int32),
        ("reserved_", C.c_int32),
    ]


class OsaParams(C.Structure):
    _fields_ = [
        ("ci", C.c_int32), ("co", C.c_int32), ("att", C.c_int32),
        ("bank", C.c_void_p),
        ("r0_w", C.c_void_p), ("r0_b", C.c_void_p), ("r2_w", C.c_void_p), ("r2_b", C.c_void_p),
        ("fc_w", C.c_void_p), ("bn_scale", C.c_void_p), ("bn_shift", C.c_void_p),
        ("ch_w", C.c_void_p), ("ch_b", C.c_void_p), ("fl_w", C.c_void_p), ("fl_b", C.c_void_p),
        ("sp_w", C.c_void_p), ("sp_b", C.c_void_p), ("kn_w", C.c_void_p), ("kn_b", C.c_void_p),
        ("pool", C.c_void_p * MAX_SRC),
        ("scratch", C.c_void_p),
        ("packed", C.c_void_p),
    ]


class SatuWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "body0_w", "body0_b", "body2_w", "body2_b", "routing_w", "routing_b", "offset_w", "offset_b",
        "st_offset_w", "st_offset_b", "compress", "expand")]


class Axpby(C.Structure):
    _fields_ = [("dst_slot", C.c_int32), ("x_slot", C.c_int32), ("y_slot", C.c_int32), ("alpha", C.c_float), ("beta", C.c_float)]


class GradPrep(C.Structure):
    _fields_ = [("dv_slot", C.c_int32), ("out_slot", C.c_int32), ("g_slot", C.c_int32), ("gt_tslot", C.c_int32),
                ("act", C.c_int32), ("slope", C.c_float),
                ("cscale", C.c_void_p), ("cscale_stride", C.c_int64),
                ("cadd", C.c_void_p), ("cadd_stride", C.c_int64), ("cadd_mul", C.c_float), ("reserved_", C.c_int32),
                ("dbias", C.c_void_p)]


class Nchw3(C.Structure):
    _fields_ = [("x_slot", C.c_int32), ("t_slot", C.c_int32)]


class PackChunk(C.Structure):
    _fields_ = [("w", C.c_void_p), ("dst", C.c_void_p), ("co_total", C.c_int32), ("ci_total", C.c_int32), ("o_base", C.c_int32),
                ("i_base", C.c_int32), ("ksize", C.c_int32), ("transposed", C.c_int32)]


class WgradItem(C.Structure):
    _fields_ = [("x_tslot", C.c_int32), ("g_tslot", C.c_int32), ("dw", C.c_void_p), ("ci_total", C.c_int32), ("ci_off", C.c_int32),
                ("o_off", C.c_int32), ("ksize", C.c_int32), ("per_sample", C.c_int32), ("layout", C.c_int32),
                ("sample_stride", C.c_int64)]


class OsaTrain(C.Structure):
    _fields_ = [("bn_weight", C.c_void_p), ("bn_bias", C.c_void_p), ("running_mean", C.c_void_p), ("running_var", C.c_void_p),
                ("momentum", C.c_float), ("eps", C.c_float), ("state", C.c_void_p), ("packed_t", C.c_void_p)]


class OsaGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "dwfold", "d_bank", "d_r0_w", "d_r0_b", "d_r2_w", "d_r2_b", "d_fc_w", "d_bn_w", "d_bn_b", "d_ch_w", "d_ch_b", "d_fl_w", "d_fl_b",
        "d_sp_w", "d_sp_b", "d_kn_w", "d_kn_b", "datt", "dvec", "dpool")]


class MaskTrain(C.Structure):
    _fields_ = ([(n, C.c_void_p) for n in ("w4", "b4", "w7", "b7", "w11", "b11")]
                + [("bn_w", C.c_void_p * 4), ("bn_b", C.c_void_p * 4), ("bn_rm", C.c_void_p * 4), ("bn_rv", C.c_void_p * 4),
                   ("gamma", C.c_void_p), ("momentum", C.c_float), ("eps", C.c_float)]
                + [(n, C.c_void_p) for n in ("m0", "t2", "m4", "t3", "m7", "t5", "m11", "mask", "stat", "sums", "coef",
                                             "d_w4", "d_b4", "d_w7", "d_b7", "d_w11", "d_b11")]
                + [("d_bn_w", C.c_void_p * 4), ("d_bn_b", C.c_void_p * 4), ("d_gamma", C.c_void_p)]
                + [(n, C.c_void_p) for n in ("dmask", "dm11", "dt4", "dm7", "dt3", "dm4", "dt2")])

MAX_TRAIN_ENTRIES = 32


# name -> (restype, argtypes); every symbol declared in include/savsr_b200.h
_VP, _I, _F, _SZ, _LL = C.c_void_p, C.c_int, C.c_float, C.c_size_t, C.c_longlong
SIGNATURES = {
    "savsr_abi_version": (_I, []),
    "savsr_last_error": (C.c_char_p, []),
    "savsr_ctx_create": (_I, [_I, C.POINTER(_VP)]),
    "savsr_ctx_destroy": (None, [_VP]),
    "savsr_ctx_sm_count": (_I, [_VP]),
    "savsr_ctx_set_format": (_I, [_VP, _I]),
    "savsr_ctx_get_format": (_I, [_VP]),
    "savsr_ctx_set_option": (_I, [_VP, _I, _I]),
    "savsr_ctx_get_option": (_I, [_VP, _I]),
    "savsr_arena_bytes": (_SZ, [_I, _I, _I, _I]),
    "savsr_arena_create": (_I, [_VP, _VP, _I, _I, _I, _I, C.POINTER(_VP)]),
    "savsr_arena_destroy": (None, [_VP]),
    "savsr_arena_tiles": (_I, [_VP]),
    "savsr_arena_import": (_I, [_VP, _I, _VP, _VP]),
    "savsr_arena_export": (_I, [_VP, _I, _VP, _VP]),
    "savsr_packed_weight_bytes": (_SZ, [_I, _I, _I]),
    "savsr_pack_conv_weight": (_I, [_VP, _I, _I, _I, _I, _I, _I, _I, _VP, _VP]),
    "savsr_conv": (_I, [_VP, _VP, C.POINTER(ConvGroup), _I, _I, _I, _I, _I, _VP]),
    "savsr_conv_wgrad": (_I, [_VP, _VP, _VP, _I, _I, _I, _I, _I, _I, _VP, _VP]),
    "savsr_slot_axpby": (_I, [_VP, _VP, C.POINTER(Axpby), _I, _VP]),
    "savsr_grad_prep": (_I, [_VP, _VP, _VP, _I, _I, C.POINTER(GradPrep), _I, _VP]),
    "savsr_slot_to_nchw3": (_I, [_VP, _VP, _VP, _I, _I, C.POINTER(Nchw3), _I, _VP]),
    "savsr_pack_conv_chunks": (_I, [_VP, _VP, _I, _I, _VP]),
    "savsr_conv_wgrad_batched": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _VP, _I, _I, _VP]),
    "savsr_adam_ema": (_I, [_VP, _VP, _VP, _VP, _VP, _VP, C.c_long, _F, _F, _F, _F, _VP, _F, _F, _VP]),
    "savsr_adam_ema_dev": (_I, [_VP, _VP, _VP, _VP, _VP, _VP, C.c_long, _VP, _F, _F, _F, _VP, _F, _F, _VP]),
    "savsr_osa_train_state_floats": (_SZ, [_I]),
    "savsr_osa_train_dvec_floats": (_SZ, [_I, _I]),
    "savsr_osa_prologue_train": (_I, [_VP, C.POINTER(OsaParams), C.POINTER(OsaTrain), _I, _I, _I, _I, _F, _F, _VP]),
    "savsr_osa_fold_backward": (_I, [_VP, C.POINTER(OsaParams), C.POINTER(OsaTrain), C.POINTER(OsaGrads), _I, _I, _VP]),
    "savsr_slot_channel_dot": (_I, [_VP, _VP, _I, _I, _VP, _VP]),
    "savsr_ca_backward": (_I, [_VP, _VP, _I, _I, _I] + [_VP] * 11 + [_VP]),
    "savsr_mask_forward_train": (_I, [_VP, _VP, C.POINTER(MaskTrain), _I, _I, _I, _I, _VP]),
    "savsr_mask_backward_train": (_I, [_VP, _VP, C.POINTER(MaskTrain), _I, _I, _I, _I, _I, _I, _VP]),
    "savsr_sta_lrelu_forward": (_I, [_VP, _VP, _VP, _VP, _I, _I, _I, _I, _F, _VP]),
    "savsr_sta_lrelu_backward": (_I, [_VP, _VP, _VP, _VP, _VP, _VP, _I, _I, _I, _I, _F, _VP]),
    "savsr_plan_create": (_I, [_VP, C.POINTER(_VP)]),
    "savsr_plan_destroy": (None, [_VP]),
    "savsr_plan_size": (_I, [_VP]),
    "savsr_plan_set_io": (_I, [_VP, _VP, _SZ, _VP, _SZ, _I]),
    "savsr_plan_set_io_u8": (_I, [_VP, _VP, _SZ, _VP, _SZ, _I]),
    "savsr_plan_set_io_u8_table": (_I, [_VP, _VP, _I, _VP, _SZ, _I]),
    "savsr_plan_set_io_u16_table": (_I, [_VP, _VP, _I, _VP, _SZ, _I]),
    "savsr_plan_add_pack_frames": (_I, [_VP, _VP, _VP, _I, _I, _I, _I]),
    "savsr_plan_add_pack_frames_u8": (_I, [_VP, _VP, _VP, _I, _I, _I, _I]),
    "savsr_plan_add_pack_frames_u8_table": (_I, [_VP, _VP, _VP, _I, _I, _I, _I]),
    "savsr_plan_add_pack_frames_u16_table": (_I, [_VP, _VP, _VP, _I, _I, _I, _I]),
    "savsr_plan_add_conv": (_I, [_VP, _VP, C.POINTER(ConvGroup), _I, _I, _I, _I, _I]),
    "savsr_plan_add_osa_prologue": (_I, [_VP, C.POINTER(OsaParams), _I, _I, _I, _I, _F, _F]),
    "savsr_plan_add_ca_scale_residual": (_I, [_VP, _VP, _I, _I, _I, _VP, _I, _VP, _VP, _VP, _VP, _VP]),
    "savsr_plan_add_osadapt_mask": (_I, [_VP, _VP, _I, _I, _I, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "savsr_plan_add_satu_kconv_sta": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _VP, _VP, _F]),
    "savsr_plan_add_satu_hr": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _I, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _I, _I, _VP]),
    "savsr_plan_add_satu_hr_u8": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _I, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _I, _I, _VP]),
    "savsr_plan_add_satu_hr_u8_table": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _I, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _I, _I, _VP]),
    "savsr_plan_add_satu_hr_u16_table": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _I, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _I, _I, _VP]),
    "savsr_plan_add_arena_export": (_I, [_VP, _VP, _I, _VP]),
    "savsr_plan_run": (_I, [_VP, _VP]),
    "savsr_forward": (_I, [_VP, _VP, _VP, _VP]),
    "savsr_forward_u8": (_I, [_VP, _VP, _VP, _VP]),
    "savsr_forward_u8_frames": (_I, [_VP, _VP, _VP, _VP]),
    "savsr_forward_u16_frames": (_I, [_VP, _VP, _VP, _VP]),
    "savsr_write_frame_table": (_I, [_VP, _VP, _VP, _I, _VP]),
    "savsr_yuv420_to_bgr": (_I, [_VP, _VP, _I, _VP, _VP, _I, _I, C.c_int64, _I, _I, _I, _VP, _VP]),
    "savsr_bgr_to_yuv420": (_I, [_VP, _VP, _I, _I, _I, _VP, _I, _VP, _VP, _I, _I, C.c_int64, _VP]),
    "savsr_yuv420_10_to_bgr48": (_I, [_VP, _VP, _I, _VP, _VP, _I, _I, C.c_int64, _I, _I, _I, _I, _VP, _VP]),
    "savsr_bgr48_to_yuv420_10": (_I, [_VP, _VP, _I, _I, _I, _VP, _I, _VP, _VP, _I, _I, C.c_int64, _I, _VP]),
    "savsr_yuv420_to_bgr_cs": (_I, [_VP, _VP, _I, _VP, _VP, _I, _I, C.c_int64, _I, _I, _I, _VP, _I, _I, _VP]),
    "savsr_bgr_to_yuv420_cs": (_I, [_VP, _VP, _I, _I, _I, _VP, _I, _VP, _VP, _I, _I, C.c_int64, _I, _I, _VP]),
    "savsr_yuv420_10_to_bgr48_cs": (_I, [_VP, _VP, _I, _VP, _VP, _I, _I, C.c_int64, _I, _I, _I, _I, _VP, _I, _I, _VP]),
    "savsr_bgr48_to_yuv420_10_cs": (_I, [_VP, _VP, _I, _I, _I, _VP, _I, _VP, _VP, _I, _I, C.c_int64, _I, _I, _I, _VP]),
    "savsr_yuv422_to_bgr_cs": (_I, [_VP, _VP, _I, _I, _VP, _VP, _I, _I, C.c_int64, _I, _I, _I, _VP, _I, _I, _VP]),
    "savsr_bgr_to_yuv422_cs": (_I, [_VP, _VP, _I, _I, _I, _VP, _I, _I, _VP, _VP, _I, _I, C.c_int64, _I, _I, _VP]),
    "savsr_yuv422_10_to_bgr48_cs": (_I, [_VP, _VP, _I, _I, _VP, _VP, _I, _I, C.c_int64, _I, _I, _I, _I, _VP, _I, _I, _VP]),
    "savsr_bgr48_to_yuv422_10_cs": (_I, [_VP, _VP, _I, _I, _I, _VP, _I, _I, _VP, _VP, _I, _I, C.c_int64, _I, _I, _I, _VP]),
    "savsr_widen_u8_to_u16": (_I, [_VP, _VP, _I, _I, _I, _VP, _VP]),
    "savsr_scene_score_u8": (_I, [_VP, _VP, _I, _I, _I, _LL, _I, _LL, _VP, _VP, _VP, _VP]),
    "savsr_scene_score_u16": (_I, [_VP, _VP, _I, _I, _I, _LL, _I, _LL, _VP, _VP, _VP, _VP]),
    "savsr_write_scene_frame_table": (_I, [_VP, _VP, _VP, _LL, _I, _VP, _LL, _I, _LL, _I, _VP]),
    "savsr_pack_frames": (_I, [_VP, _VP, _VP, _I, _I, _I, _I, _VP]),
    "savsr_pack_frames_u8": (_I, [_VP, _VP, _VP, _I, _I, _I, _I, _VP]),
    "savsr_pack_frames_u8_table": (_I, [_VP, _VP, _VP, _I, _I, _I, _I, _VP]),
    "savsr_pack_frames_u16_table": (_I, [_VP, _VP, _VP, _I, _I, _I, _I, _VP]),
    "savsr_osa_prologue": (_I, [_VP, C.POINTER(OsaParams), _I, _I, _I, _I, _F, _F, _VP]),
    "savsr_ca_scale_residual": (_I, [_VP, _VP, _I, _I, _I, _VP, _I, _VP, _VP, _VP, _VP, _VP, _VP]),
    "savsr_osadapt_mask": (_I, [_VP, _VP, _I, _I, _I, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "savsr_satu_index": (_I, [_VP, C.POINTER(SatuWeights), _I, _I, _I, _I, _F, _F] + [_VP] * 9 + [_VP]),
    "savsr_satu_kconv_sta": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _VP, _VP, _F, _VP]),
    "savsr_satu_hr": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _I, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _I, _I, _VP, _VP]),
    "savsr_satu_hr_u8": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _I, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _I, _I, _VP, _VP]),
    "savsr_satu_hr_u8_table": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _I, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _I, _I, _VP, _VP]),
    "savsr_satu_hr_u16_table": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _I, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _I, _I, _VP, _VP]),
    "savsr_img_metrics_blocks": (_I, [_VP, _I, _I]),
    "savsr_img_metrics": (_I, [_VP, _VP, _VP, _I, _I, _I, _VP, _VP, _VP]),
    "savsr_ssim_y_blocks": (_I, [_I, _I]),
    "savsr_ssim_y": (_I, [_VP, _VP, _VP, _I, _I, _I, _VP, _VP]),
    "savsr_aa_max_taps": (_I, [_I, _I]),
    "savsr_aa_table": (_I, [_VP, _I, _I, _I, _VP, _VP, _VP, _VP, _VP]),
    "savsr_lr_synthesize": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _I, _I, _VP, _VP, _VP, _I, _VP, _VP, _VP, _I, _VP, _VP, _VP, _VP]),
    "savsr_resize_aa": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _VP, _VP, _VP, _I, _VP, _VP, _VP, _I, _VP, _VP, _VP]),
}

_lib: Optional[C.CDLL] = None


def load() -> C.CDLL:
    """Load the shared library and bind every declared symbol.  Raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SavsrError(
            f"{LIB_PATH} not found: build it with `python -m savsr_b200.build` (needs nvcc, sm_100a). "
            "savsr_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.savsr_abi_version() != ABI_VERSION:
        raise SavsrError(f"ABI version mismatch: library {lib.savsr_abi_version()}, binding {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().savsr_last_error()
        raise SavsrError(f"libsavsr_sm100 error {rc}: {msg.decode(errors='replace') if msg else '?'}")


class Context:
    """savsr_ctx wrapper (one per device)."""

    def __init__(self, device: int):
        self.lib = load()
        h = C.c_void_p()
        check(self.lib.savsr_ctx_create(int(device), C.byref(h)))
        self.handle = h
        self.device = int(device)
        self.sm_count = self.lib.savsr_ctx_sm_count(h)

    def set_option(self, option: int, value: int) -> None:
        check(self.lib.savsr_ctx_set_option(self.handle, int(option), int(value)))

    def set_format(self, fmt: int) -> None:
        """16-bit storage / operand format (FMT_BF16 or FMT_FP16) used by every later call on this context."""
        check(self.lib.savsr_ctx_set_format(self.handle, int(fmt)))

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.savsr_ctx_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class Arena:
    """savsr_arena wrapper over caller-owned device memory (`base_ptr`)."""

    def __init__(self, ctx: Context, base_ptr: int, nslots: int, batch: int, height: int, width: int):
        self.ctx = ctx
        self.lib = ctx.lib
        h = C.c_void_p()
        check(self.lib.savsr_arena_create(ctx.handle, C.c_void_p(base_ptr), nslots, batch, height, width, C.byref(h)))
        self.handle = h
        self.nslots, self.batch, self.height, self.width = nslots, batch, height, width
        self.tiles = self.lib.savsr_arena_tiles(h)

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.savsr_arena_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class CPlan:
    """savsr_plan wrapper: the recorded launch list of one forward, replayed by one C call."""

    def __init__(self, ctx: Context):
        self.lib = ctx.lib
        h = C.c_void_p()
        check(self.lib.savsr_plan_create(ctx.handle, C.byref(h)))
        self.handle = h

    def __len__(self) -> int:
        return int(self.lib.savsr_plan_size(self.handle))

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.savsr_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass
