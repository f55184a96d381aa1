/*
 * savsr_b200.h -- C ABI of libsavsr_sm100.so: the B200 (sm_100a) kernels behind the SAVSR forward
 * hot path (OSA-Conv + bi-directional propagation trunk + SATU upsampler).
 *
 * The reference (Weepingchestnut/SAVSR) has no C ABI of its own: its hot path is the Python file
 * lbasicsr/archs/savsr_arch.py calling ATen ops.  Every entry point below therefore cites the
 * reference *Python* interface it replaces (file:line relative to the reference root); the
 * binding a maintainer would add on the reference side is the ctypes stub in INTEGRATION.md
 * (savsr_b200/_capi.py is that stub, shipped).
 *
 * Conventions (mirroring the reference's native-op idiom, ops/fused_act/src/fused_bias_act.cpp:10-26):
 *   - plain pointers and sizes only; no torch types.  All pointers are DEVICE pointers unless noted.
 *   - the caller owns and allocates every buffer (inputs, outputs, activation arenas, scratch).
 *     The library never allocates device memory, never synchronises, and launches only on the
 *     stream it is given (so every call is CUDA-graph capturable).  It holds no process-wide mutable
 *     state: everything lives in the savsr_ctx (one per device); launchers switch to the context's
 *     device for the duration of the call and restore the caller's current device.
 *   - every function returns 0 on success, non-zero on error; savsr_last_error() returns a
 *     thread-local message.  A device without sm_100 tensor-core support is an error, never a
 *     fallback.
 *   - activations live in an "arena": bf16, NHWC with C = 64, shape [nslots * batch, H, W, 64];
 *     "slot s, sample n" is image index s * batch + n.  A 64*k-channel tensor is k slots.
 */
#ifndef SAVSR_B200_H_
#define SAVSR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SAVSR_ABI_VERSION 4
#define SAVSR_MAX_SRC 5      /* most 64-channel sources one conv concatenates (OSA 320->64)      */
#define SAVSR_MAX_GROUPS 25  /* most independent convolutions batched into one launch            */
#define SAVSR_TILE_W 8       /* output tile = 8 x 16 pixels = 128 GEMM rows (one UMMA M)         */
#define SAVSR_TILE_H 16

typedef struct savsr_ctx savsr_ctx;     /* per-device context (driver entry points, SM count)   */
typedef struct savsr_arena savsr_arena; /* activation arena + its TMA descriptors               */
typedef void* savsr_stream;             /* cudaStream_t                                          */

/* 16-bit storage / tensor-core operand format of arenas and packed weights (accumulation is always fp32).
 * BF16: the throughput path named by the task (<= 0.05 dB PSNR delta).  FP16: same speed, 10-bit mantissa: the
 * high-precision path that meets the <= 1e-3 max-abs bound; activations must stay below 65504. */
enum savsr_format { SAVSR_FMT_BF16 = 0, SAVSR_FMT_FP16 = 1 };
/* Row (output channel) order inside a packed n_tile = 64 weight block.  LINEAR: row n = channel n.  QUAD: row n =
 * channel with the bit fields [2:1] and [4:3] of n swapped -- the order savsr_conv requires for n_tile 64 (its epilogue
 * reads the accumulator with 16x256b TMEM loads and stores 16 contiguous bytes per thread), savsr_satu_kconv_sta likewise. */
enum savsr_row_order { SAVSR_ROWS_LINEAR = 0, SAVSR_ROWS_QUAD = 1 };

enum savsr_act { SAVSR_ACT_NONE = 0, SAVSR_ACT_LRELU = 1, SAVSR_ACT_RELU = 2 };

/* how a convolution writes its result */
enum savsr_dst_mode {
  SAVSR_DST_ARENA = 0, /* bf16 NHWC-64 arena slot (N = 64)                                       */
  SAVSR_DST_AUX16 = 1  /* fp32 [batch][H*W][16] side buffer (N = 16; OSAdapt mask conv)          */
};

enum savsr_conv_impl {
  SAVSR_IMPL_TCGEN05_TAP = 0,  /* tcgen05/TMEM implicit GEMM, one TMA box per filter tap          */
  SAVSR_IMPL_TCGEN05_HALO = 1, /* same, one halo box per source reused by all nine taps            */
  SAVSR_IMPL_CHECK = 2         /* slow CUDA-core kernel, same contract: on-device checker only     */
};

/*
 * One convolution of a batched launch.  Replaces one nn.Conv2d / F.conv2d call of
 * savsr_arch.py (388-397 ResidualBlock convs, 429-442 WindowUnit_l1, 480-483 WindowUnit_l2,
 * 541-543 RCAB, 567 ResidualGroup.conv, 166 OSA-Conv grouped conv, 190 OSAdapt mask,
 * 620 h_win_conv_h, 629 conv_last) together with the
 * torch.cat feeding it (404, 412, 462, 498, 721, 374) and the elementwise ops that follow it.
 *
 *   acc = sum_{s < nsrc} sum_{tap} W[s, tap] * src_s(shifted by tap)          (zero padding)
 *   v   = act(acc + bias) ; v *= mask[pixel] ; v += res1 ; v += res2_scale * res2 ; store v      (LeakyReLU slope in [0, 1])
 *   pool (optional): per-(sample, tile-warp) partial channel sums of v, consumed by the next
 *   OSA-Conv / channel-attention global average pool (savsr_arch.py:146, 515).
 */
typedef struct savsr_conv_group {
  int32_t src_slot[SAVSR_MAX_SRC];
  int32_t nsrc;
  int32_t dst_slot;             /* SAVSR_DST_ARENA only                                          */
  int32_t res1_slot;            /* -1 = none                                                     */
  int32_t res2_slot;            /* -1 = none                                                     */
  float res2_scale;
  int32_t act;                  /* enum savsr_act                                                */
  float slope;                  /* LeakyReLU negative slope                                      */
  const void* weight;           /* packed bf16, see savsr_pack_conv_weight                       */
  int64_t weight_sample_stride; /* BYTES between per-sample weights (OSA-Conv); 0 = shared       */
  const float* bias;            /* [N] fp32 or NULL                                              */
  const float* mask;            /* [batch][H*W] fp32 per-pixel multiplier or NULL (OSAdapt)      */
  float* pool;                  /* [batch][tiles*4][64] fp32 partial sums or NULL                */
  void* aux_dst;                /* SAVSR_DST_AUX16 destination                                   */
  int32_t src_channels;         /* 0 (= 64) or 16 / 32 / 48: only this many LEADING channels of every source carry data, the
                                   rest are zero in the arena AND in the filter (first layer: 21 frame channels of 64); the
                                   tensor-core K loop skips the zero part.  Same value for all groups of a launch.          */
  int32_t reserved_;
} savsr_conv_group;

/* Tuning / bring-up knobs of a context (savsr_ctx_set_option).  The library reads no environment variables. */
enum savsr_option {
  SAVSR_OPT_BIGK_ALL = 0,     /* 1 (default): every 3x3 HALO N=64 conv runs on the batched dual-issuer kernel; 0: only K > 18 blocks */
  SAVSR_OPT_BIGK_ISSUERS = 1, /* MMA-issuing warps of that kernel: 2 (default) or 1                                                  */
  SAVSR_OPT_PDL = 2,          /* 1: launch with programmatic stream serialization (the next kernel's CTAs start while this one drains and
                                 block in griddepcontrol.wait before touching memory); pays for chains of microsecond-sized launches
                                 (training at 4 x 64 x 64), not for long ones.  Default 0                                                */
  SAVSR_OPT_COUNT = 3
};

/* ---- library / context ------------------------------------------------------------------- */
int savsr_abi_version(void);
const char* savsr_last_error(void);
/* Fails unless `device` is compute capability 10.x (tcgen05 / TMEM / TMA present). */
int savsr_ctx_create(int device, savsr_ctx** out);
void savsr_ctx_destroy(savsr_ctx* ctx);
int savsr_ctx_sm_count(const savsr_ctx* ctx);
/* Select the 16-bit format used by every later call on this context (default SAVSR_FMT_BF16). */
int savsr_ctx_set_format(savsr_ctx* ctx, int format);
int savsr_ctx_get_format(const savsr_ctx* ctx);
/* option: enum savsr_option.  Returns non-zero for an unknown option or an out-of-range value. */
int savsr_ctx_set_option(savsr_ctx* ctx, int option, int value);
int savsr_ctx_get_option(const savsr_ctx* ctx, int option);

/* ---- activation arenas --------------------------------------------------------------------- */
/* Bytes the caller must allocate (256-byte aligned) for an arena of that shape. */
size_t savsr_arena_bytes(int nslots, int batch, int height, int width);
int savsr_arena_create(savsr_ctx* ctx, void* base, int nslots, int batch, int height, int width,
                       savsr_arena** out);
void savsr_arena_destroy(savsr_arena* a);
int savsr_arena_tiles(const savsr_arena* a);             /* output tiles per image                */
/* debug / test helpers: fp32 NCHW [batch][64][H][W] <-> arena slot */
int savsr_arena_import(savsr_arena* a, int slot, const float* nchw, savsr_stream st);
int savsr_arena_export(savsr_arena* a, int slot, float* nchw, savsr_stream st);

/* ---- weights --------------------------------------------------------------------------------- */
/* Packed size in bytes of a [co][ci][k][k] filter (co multiple of n_tile, ci multiple of 64). */
size_t savsr_packed_weight_bytes(int co, int ci, int ksize);
/*
 * fp32 OIHW [co][ci][k][k] (k = 1 or 3) -> bf16 blocks [co/n_tile][ci/64 * k*k][n_tile][64] in the
 * 128-byte-swizzled K-major layout tcgen05.mma reads (block index = source * k*k + ky*k + kx).
 * co_real <= co rows are read, the rest are zero (tail conv: 3 -> 16).  n_tile is 64 or 16.
 * row_order (enum savsr_row_order) applies to n_tile 64 only; n_tile 16 blocks are always LINEAR.
 */
int savsr_pack_conv_weight(const float* w_oihw, int co_real, int co, int ci, int ksize, int n_tile,
                           int format /* enum savsr_format */, int row_order /* enum savsr_row_order */,
                           void* packed, savsr_stream st);

/* ---- convolutions (tensor-core hot path) ------------------------------------------------------- */
/*
 * Batched implicit-GEMM convolution: `ngroups` independent convs x `batch` samples in one launch.
 * ksize 3 (pad 1) or 1.  n_tile = 64 (dst ARENA) or 16 (AUX16).
 */
int savsr_conv(savsr_ctx* ctx, savsr_arena* arena, const savsr_conv_group* groups, int ngroups,
               int ksize, int n_tile, int dst_mode, int impl, savsr_stream st);

/*
 * First layer (savsr_arch.py:456-457 conv_sup / conv_c with the frame gather of 447-454): pack the fp32 window into ONE
 * arena slot (channel 3f+c = frame f, colour c; remaining channels zero; reflect pad of savsr_arch.py:670-690 fused),
 * after which conv_c / conv_sup are ordinary savsr_conv launches with zero-expanded [64][64][3][3] weights.
 */
int savsr_pack_frames(savsr_ctx* ctx, savsr_arena* arena, const float* x, int t, int h, int w, int dst_slot,
                      savsr_stream st);
/*
 * The same from a decoded 8-bit window: x uint8 [batch][t][h][w][3], BGR (the layout cv2.imread and video decoders produce).
 * Each value becomes float(u) / 255 correctly rounded (the reference's img.astype(np.float32) / 255.) with channels swapped to RGB,
 * so the slot is bit-identical to savsr_pack_frames of that fp32 window.
 */
int savsr_pack_frames_u8(savsr_ctx* ctx, savsr_arena* arena, const uint8_t* x, int t, int h, int w, int dst_slot,
                         savsr_stream st);
/*
 * The same from a frame table: frames is a DEVICE array const uint8_t* [batch][t] (savsr_write_frame_table), and entry n * t + f points
 * at frame f of sample n, one contiguous uint8 [h][w][3] BGR frame.  The slot is bit-identical to savsr_pack_frames_u8 of the window
 * those frames would form.  Frames may repeat and may lie anywhere on the context's device (a ring of decoded frames, read in place).
 * Ownership: the table and every frame it points at must stay valid, in stream order, until the launch that reads them has run.
 */
int savsr_pack_frames_u8_table(savsr_ctx* ctx, savsr_arena* arena, const uint8_t* const* frames, int t, int h, int w, int dst_slot,
                               savsr_stream st);
/*
 * The same from a table of 16-bit frames: entry n * t + f points at one contiguous uint16 [h][w][3] BGR frame (bgr48, full scale
 * 65535), and each value v becomes float(v) / 65535 correctly rounded.  An 8-bit frame widened by 257 gives the slot its 8-bit
 * original gives.  The table holds frame addresses like the 8-bit one and is written by savsr_write_frame_table; same ownership rule.
 */
int savsr_pack_frames_u16_table(savsr_ctx* ctx, savsr_arena* arena, const uint16_t* const* frames, int t, int h, int w, int dst_slot,
                                savsr_stream st);
/*
 * Frame table writer: table_dev[i] = ptrs_host[i] for i < n, on stream st.  The pointers travel in the launches' by-value arguments
 * (448 per launch, more launches above that), never through a host-to-device copy, so the call returns at once and can be enqueued
 * in stream order in front of a graph replay that reads the table.  Refuses a null entry before any launch.
 */
int savsr_write_frame_table(savsr_ctx* ctx, const uint8_t** table_dev, const uint8_t* const* ptrs_host, int n, savsr_stream st);

/* ---- backward of the 3x3 convolution (next row 8f1: training step, lbasicsr/models/sr_model.py:101-128) ----------------------
 * Data gradient: a 3x3 convolution of dY with the transposed, spatially flipped filter -- call savsr_conv with those weights
 * (savsr_b200/autograd.py does).  Weight gradient, on tcgen05 with the pixel index as the contraction dimension:
 *   dW[o][i][ky][kx] += sum_{n, p} dY[n][o][p] * X[n][i][p + (ky-1, kx-1)]                     (zero padding)
 * dy_nchw16: 16-bit (context format) NCHW tensor [batch][64][height][pitch], pitch a multiple of 8 elements, pixels [width, pitch)
 * of every row ZERO.  x3_nchw16: [3][batch][ci][height][pitch], ci = 64, 128, ... 320: X shifted along x by -1, 0, +1 pixel
 * (copy d holds X[.., x + d - 1], zero where that leaves the row) -- TMA boxes start on 16-byte granules, so the one-pixel shifts of
 * the contraction operand are materialised by the caller.  dw: fp32 [64][ci][3][3] (per_sample = 0) or
 * [batch][64][ci][3][3] (per_sample = 1: the per-sample folded kernels of OSA-Conv), accumulated with atomics: zero it first.
 */
int savsr_conv_wgrad(savsr_ctx* ctx, const void* x3_nchw16, const void* dy_nchw16, int batch, int ci, int height, int width,
                     int pitch, int per_sample, float* dw, savsr_stream st);

/* ---- native training step (row 8f1, stage B) ---------------------------------------------------------------------------------
 * The reference's optimisation step (lbasicsr/models/sr_model.py:101-128: forward, Charbonnier, autograd backward through cuDNN
 * dgrad / wgrad, Adam; base_model.py:75-82 EMA) as launches on the activation arena.  Gradients of activations live in slots of
 * the same arena; the weight gradient reads pixel-contiguous copies from a second caller-owned buffer, the "T-arena":
 * 16-bit NCHW, T-slot t = [batch][64][height][pitch] (pitch = width rounded up to a multiple of 8; allocate it zeroed: the gradient
 * copies keep their padding columns zero, which is what makes the padded contraction exact -- the right-shifted activation copy may
 * carry one pixel into its first padding column).  savsr_b200/trainplan.py drives them.
 * Every `entries` array below is HOST memory (copied into the launch), at most 32 entries per call; `*_dev` arrays are DEVICE memory.
 */
typedef struct savsr_axpby {
  int32_t dst_slot, x_slot, y_slot;   /* y_slot -1: dst = alpha * x                                              */
  float alpha, beta;                  /* dst = alpha * x + beta * y (dst may alias x or y)                       */
} savsr_axpby;
int savsr_slot_axpby(savsr_ctx* ctx, savsr_arena* arena, const savsr_axpby* entries, int n, savsr_stream st);

/* Gradient entering a convolution whose epilogue was v = act(acc + bias) (+ pooled mean taken from v):
 *   g = (dV * cscale[n][c] + cadd_mul * cadd[n][c]) * act'(out)       act' from the sign of the stored output
 * written to g_slot (NHWC, operand of the data gradient; may equal dv_slot), to T-slot gt_tslot (operand of the weight
 * gradient) and summed over (n, y, x) into dbias (+=).  cscale: RCAB channel attention (savsr_arch.py:547-549); cadd: the
 * gradient of a global average pool of the output (OSA-Conv / channel attention inputs, savsr_arch.py:146, 515). */
typedef struct savsr_grad_prep_entry {
  int32_t dv_slot, out_slot, g_slot, gt_tslot;   /* g_slot / gt_tslot -1: not written                            */
  int32_t act;                                   /* enum savsr_act of the forward epilogue                       */
  float slope;
  const float* cscale; int64_t cscale_stride;    /* [batch][stride] fp32, 64 used; NULL = 1                      */
  const float* cadd; int64_t cadd_stride; float cadd_mul;   /* NULL = 0                                          */
  int32_t reserved_;
  float* dbias;                                  /* [64] fp32 or NULL                                            */
} savsr_grad_prep_entry;
int savsr_grad_prep(savsr_ctx* ctx, savsr_arena* arena, void* tbase, int ntslots, int pitch, const savsr_grad_prep_entry* entries, int n,
                    savsr_stream st);

/* Arena slot -> T-slots t_slot, t_slot + 1, t_slot + 2 = the activation shifted along x by -1, 0, +1 pixel (copy d holds
 * X[.., x + d - 1], zero outside the row): TMA boxes start on 16-byte granules, so the shifts are materialised. */
typedef struct savsr_nchw3 { int32_t x_slot, t_slot; } savsr_nchw3;
int savsr_slot_to_nchw3(savsr_ctx* ctx, savsr_arena* arena, void* tbase, int ntslots, int pitch, const savsr_nchw3* entries, int n,
                        savsr_stream st);

/* One (64 output channels x 64 input channels) corner of an fp32 OIHW filter [co_total][ci_total][k][k] -> k*k tensor-core blocks
 * [64][64] (16-bit, context format, SAVSR_ROWS_QUAD, 128-byte swizzle; k*k*8192 bytes at dst).  transposed = 0: rows = output
 * channels o_base.., K = input channels i_base.. (forward operand: block (source s, tap) of savsr_pack_conv_weight).
 * transposed = 1: rows = input channels, K = output channels, taps flipped: the operand of the data gradient
 * dX = conv(dY, W^T flipped).  Channels beyond co_total / ci_total read as zero. */
typedef struct savsr_pack_chunk {
  const float* w;
  void* dst;
  int32_t co_total, ci_total, o_base, i_base, ksize, transposed;
} savsr_pack_chunk;
int savsr_pack_conv_chunks(savsr_ctx* ctx, const savsr_pack_chunk* chunks_dev, int first, int count, savsr_stream st);

/* Weight gradients of many convolutions in one persistent tcgen05 launch (the kernel of savsr_conv_wgrad, table-driven).
 * Item = one (convolution, 64-channel source):   dw[(o_off + o) * ci_total + ci_off + i][tap] += sum_{n,p} g[n][o][p] x[n][i][p + tap]
 * x_tslot: first of the source's three shifted T-slots (savsr_slot_to_nchw3); g_tslot: the T-slot savsr_grad_prep wrote.
 * ksize 3: dw is [..][ci_total][3][3]; ksize 1: [..][ci_total] (centre tap).  per_sample: dw advances sample_stride floats per
 * sample (the folded kernels of OSA-Conv).  dw is accumulated with atomics: zero it first. */
enum savsr_wgrad_layout {
  SAVSR_WGRAD_OIHW = 0, /* dw[o][i][ky][kx]: the parameter's own layout (scalar atomics)                                     */
  SAVSR_WGRAD_TIO = 1   /* dw[tap][i][64]: output channels contiguous, 16-byte vector atomics (4x fewer reductions); used for the
                           per-sample gradients of OSA-Conv's folded kernels, whose only reader is savsr_osa_fold_backward; ksize 3, co 64 */
};
typedef struct savsr_wgrad_item {
  int32_t x_tslot, g_tslot;
  float* dw;
  int32_t ci_total, ci_off, o_off, ksize, per_sample, layout;
  int64_t sample_stride;
} savsr_wgrad_item;
int savsr_conv_wgrad_batched(savsr_ctx* ctx, const void* tbase, int ntslots, int batch, int height, int width, int pitch,
                             const savsr_wgrad_item* items_dev, int first, int count, savsr_stream st);

/* torch.optim.Adam (no weight decay, no amsgrad; sr_model.py:77-89, train YAML lr 2e-4, betas 0.9 / 0.99) followed by the EMA of
 * base_model.py:75-82, over flat fp32 buffers.  step_dev: device scalar holding the step count t >= 1 as a float (bias corrections
 * 1 - beta^t).  grad_scale multiplies the gradient first (1 / world size after a summing all-reduce).  ema may be NULL. */
int savsr_adam_ema(savsr_ctx* ctx, float* param, const float* grad, float* exp_avg, float* exp_avg_sq, float* ema, long n, float lr,
                   float beta1, float beta2, float eps, const float* step_dev, float ema_decay, float grad_scale, savsr_stream st);
/* savsr_adam_ema with the learning rate read from device memory (lr_dev: one float, read when the kernel starts), so a captured CUDA
 * graph follows a schedule that rewrites *lr_dev between replays.  Same arithmetic: bit-identical to savsr_adam_ema at the same lr. */
int savsr_adam_ema_dev(savsr_ctx* ctx, float* param, const float* grad, float* exp_avg, float* exp_avg_sq, float* ema, long n,
                       const float* lr_dev, float beta1, float beta2, float eps, const float* step_dev, float ema_decay, float grad_scale,
                       savsr_stream st);

/* ---- OSA-Conv prologue (savsr_arch.py:143-163, 91-96, 123-128) ---------------------------------- */
typedef struct savsr_osa_params {
  int32_t ci, co, att;            /* in planes (64*nsrc), out planes (64), attention channels      */
  const float* bank;              /* [8][co][ci][3][3] fp32 weight bank                            */
  const float* r0_w; const float* r0_b;   /* scale_routing.0  [2ci][ci+2], [2ci]                  */
  const float* r2_w; const float* r2_b;   /* scale_routing.2  [ci][2ci],   [ci]                   */
  const float* fc_w;                      /* attention.fc     [att][ci]                            */
  const float* bn_scale; const float* bn_shift; /* eval BatchNorm folded to z*scale+shift, [att]  */
  const float* ch_w; const float* ch_b;   /* channel_fc [ci][att], [ci]                            */
  const float* fl_w; const float* fl_b;   /* filter_fc  [co][att], [co]                            */
  const float* sp_w; const float* sp_b;   /* spatial_fc [9][att],  [9]                             */
  const float* kn_w; const float* kn_b;   /* kernel_fc  [8][att],  [8]                             */
  const float* pool[SAVSR_MAX_SRC];       /* per source: [batch][npart][64] partial sums           */
  float* scratch;                         /* [batch][5*ci + 192] fp32 work area                    */
  void* packed;                           /* out: [batch] packed bf16 weights (n_tile 64)          */
} savsr_osa_params;
/*
 * For each OSA-Conv of the launch and each sample: global-average-pool vector (from the producers'
 * partial sums) -> scale_routing MLP -> ScaleAttention heads -> per-sample modulated kernel
 * W'[o,i,u,v] = fa[o] ca[i] sa[u,v] sum_k ka[k] bank[k,o,i,u,v], written packed for savsr_conv.
 * inv_scale_h/w = 1/s_h, 1/s_w (fp32).  npart = partial sums per image, npix = H*W of the pool.
 */
int savsr_osa_prologue(savsr_ctx* ctx, const savsr_osa_params* convs, int nconvs, int batch,
                       int npart, int npix, float inv_scale_h, float inv_scale_w, savsr_stream st);
/* test hook: per sample, scratch + 4*ci + 8 holds the attention vectors [ca(ci) | fa(co) | sa(9) | ka(8)] */

/* Train-mode OSA-Conv prologue (savsr_arch.py:139-163 with ScaleAttention's BatchNorm on BATCH statistics, as nn.BatchNorm2d does
 * in train mode: biased variance normalises, running statistics move by `momentum` with the unbiased variance) and its backward.
 * convs[i] as for savsr_osa_prologue (bn_scale / bn_shift unused; scratch must be private to this convolution: it keeps the
 * forward's intermediate vectors for the backward); batch <= 32.  Besides convs[i].packed (forward operand, [n][s][9][64][64]) the
 * folded kernels are also written transposed + flipped (data-gradient operand) to extra[i].packed_t as [s][n][9][64][64]. */
typedef struct savsr_osa_train {
  const float* bn_weight; const float* bn_bias;   /* [att]                                                        */
  float* running_mean; float* running_var;        /* [att], updated in place; both NULL = not tracked             */
  float momentum, eps;
  float* state;                                   /* savsr_osa_train_state_floats(batch) floats, kept for backward */
  void* packed_t;
} savsr_osa_train;
/* Gradient side of one OSA-Conv.  dwfold: fp32 [batch][64][ci][3][3] weight gradient of the folded kernels (from
 * savsr_conv_wgrad_batched, per_sample) -- consumed AND zeroed.  d_*: gradients of the parameters, accumulated (+=).
 * datt: [batch][ci + 64 + 17] scratch, zero on entry, left zero.  dvec: savsr_osa_train_dvec_floats(batch, ci) floats scratch.
 * dpool: out [batch][ci] = gradient of the pooled means (savsr_grad_prep cadd of the producing convolutions). */
typedef struct savsr_osa_grads {
  float* dwfold;
  float* d_bank;
  float* d_r0_w; float* d_r0_b; float* d_r2_w; float* d_r2_b;
  float* d_fc_w; float* d_bn_w; float* d_bn_b;
  float* d_ch_w; float* d_ch_b; float* d_fl_w; float* d_fl_b; float* d_sp_w; float* d_sp_b; float* d_kn_w; float* d_kn_b;
  float* datt; float* dvec; float* dpool;
} savsr_osa_grads;
size_t savsr_osa_train_state_floats(int batch);
size_t savsr_osa_train_dvec_floats(int batch, int ci);
int savsr_osa_prologue_train(savsr_ctx* ctx, const savsr_osa_params* convs, const savsr_osa_train* extra, int nconvs, int batch,
                             int npart, int npix, float inv_scale_h, float inv_scale_w, savsr_stream st);
int savsr_osa_fold_backward(savsr_ctx* ctx, const savsr_osa_params* convs, const savsr_osa_train* extra, const savsr_osa_grads* grads,
                            int nconvs, int batch, savsr_stream st);

/* Backward of the RCAB channel attention dst = x + t * y, y = sigmoid(W2 relu(W1 mean(t) + b1) + b2) (savsr_arch.py:514-524):
 * savsr_slot_channel_dot: out[n][c] += sum_p a[n,p,c] b[n,p,c] over two arena slots (dy = <dout, t>; out zero on entry);
 * savsr_ca_backward: from dy (consumed and zeroed) and the saved y: parameter gradients (+=) and dmean [batch][64], the gradient of
 * the pooled mean; the gradient of t itself is dout * y + dmean / npix (savsr_grad_prep cscale / cadd). */
int savsr_slot_channel_dot(savsr_ctx* ctx, savsr_arena* arena, int a_slot, int b_slot, float* out, savsr_stream st);
int savsr_ca_backward(savsr_ctx* ctx, const float* pool, int npart, int npix, int batch, const float* w1, const float* b1, const float* w2,
                      const float* b2, const float* y, float* dy, float* dw1, float* db1, float* dw2, float* db2, float* dmean,
                      savsr_stream st);

/* Train-mode OSAdapt mask net + combination (savsr_arch.py:186-214, 727-732), everything after the 64 -> 16 convolution:
 *   m0 (from savsr_conv, N = 16, no activation) -> BN1 -> ReLU -> AvgPool2 -> conv4 -> BN5 -> ReLU -> conv7 -> BN8 -> ReLU -> bilinear x2
 *   -> conv11 -> BN12 -> sigmoid = mask ;   out = R + a * mask + gamma * share           (a = OSA-Conv(R); R, a, share, out: arena slots)
 * BatchNorm on batch statistics (indices 0..3 = BN1, BN5, BN8, BN12), running statistics updated in place when given.  All maps are
 * fp32 channel-last: m0, t5 [batch][H*W][16]; t2, m4, t3, m7 [batch][(H/2)*(W/2)][16]; m11, mask [batch][H*W]; they stay alive for the
 * backward.  stat: 4 x 32 floats (mean | rstd per layer); sums: 64 doubles of scratch, zero on entry, left zero; coef: 4 x 48 floats.
 * savsr_mask_backward_train: from the gradient of `out` (dh_slot): da_slot = dh * mask, gshare_slot = gamma * dh (the caller accumulates
 * them and dh itself into the gradients of a, share and R), the gradients of every parameter of the mask net and of gamma (+=), and the
 * gradient of m0 as the first 16 channels of arena slot dm0_slot (channels 16..63 are not written: keep them zero) -- the operand of the
 * tensor-core data / weight gradient of the 64 -> 16 convolution.  dmask .. dt2: scratch of the sizes of mask, m11, t2 (x5). */
typedef struct savsr_mask_train {
  const float *w4, *b4, *w7, *b7, *w11, *b11;
  const float* bn_w[4]; const float* bn_b[4];
  float* bn_rm[4]; float* bn_rv[4];
  const float* gamma;
  float momentum, eps;
  float *m0, *t2, *m4, *t3, *m7, *t5, *m11, *mask;
  float* stat; double* sums; float* coef;
  float *d_w4, *d_b4, *d_w7, *d_b7, *d_w11, *d_b11;
  float* d_bn_w[4]; float* d_bn_b[4];
  float* d_gamma;
  float *dmask, *dm11, *dt4, *dm7, *dt3, *dm4, *dt2;
} savsr_mask_train;
int savsr_mask_forward_train(savsr_ctx* ctx, savsr_arena* arena, const savsr_mask_train* m, int r_slot, int a_slot, int share_slot, int out_slot,
                             savsr_stream st);
int savsr_mask_backward_train(savsr_ctx* ctx, savsr_arena* arena, const savsr_mask_train* m, int dh_slot, int a_slot, int share_slot, int da_slot,
                              int gshare_slot, int dm0_slot, savsr_stream st);

/* sta_conv of STAUpsample fused with kernel_conv's LeakyReLU, for the training step (savsr_arch.py:297-313, 226-228), fp32 NCHW:
 *   out[b,c,p] = sum_{t<25} x[b,c,clamp(p + d_t)] * lrelu(kpre[b, c*25 + t, p])     (replicate padding; t = 5 u + v, d_t = (u - 2, v - 2))
 * x, out, dout, dx: [batch][channels][height][width]; kpre, dkpre: [batch][channels*25][height][width] (the output of kernel_conv BEFORE
 * its activation).  backward writes dx and dkpre (no accumulation). */
int savsr_sta_lrelu_forward(savsr_ctx* ctx, const float* x, const float* kpre, float* out, int batch, int channels, int height, int width,
                            float slope, savsr_stream st);
int savsr_sta_lrelu_backward(savsr_ctx* ctx, const float* x, const float* kpre, const float* dout, float* dx, float* dkpre, int batch, int channels,
                             int height, int width, float slope, savsr_stream st);

/* ---- RCAB channel attention (savsr_arch.py:514-524, 547-549) --------------------------------------
 * y = sigmoid(W2 relu(W1 mean(t) + b1) + b2) ; dst = x + t * y        (t, x, dst: arena slots)
 * Two launches: the per-sample channel-scale vector, then the streaming pass.                      */
int savsr_ca_scale_residual(savsr_ctx* ctx, savsr_arena* arena, int t_slot, int x_slot, int dst_slot,
                            const float* pool, int npart, const float* w1, const float* b1,
                            const float* w2, const float* b2, float* y_scratch /* [batch][64] */, savsr_stream st);

/* ---- OSAdapt mask tail (savsr_arch.py:193-205) ------------------------------------------------------
 * in16: [batch][H*W][16] fp32 = ReLU(BN(conv64->16(x))) from savsr_conv(AUX16).  Runs AvgPool2d(2),
 * two conv16->16+BN+ReLU at half resolution, bilinear x2 upsample, conv16->1+BN, sigmoid.
 * Weights: BN already folded by the caller.  wa/wb: [16][16][3][3], wc: [1][16][3][3].
 * half0/half1: [batch][(H/2)*(W/2)][16] fp32 scratch (half1 receives the nine per-tap projections of the last conv,
 * which commutes with the upsample; contents are internal).  mask out: [batch][H*W] fp32.            */
int savsr_osadapt_mask(savsr_ctx* ctx, const float* in16, int batch, int height, int width,
                       const float* wa, const float* ba, const float* wb, const float* bb,
                       const float* wc, const float* bc, float* half0, float* half1, float* mask,
                       savsr_stream st);

/* ---- SATU (savsr_arch.py:315-376, 262-313) ---------------------------------------------------------- */
typedef struct savsr_satu_weights {
  const float* body0_w; const float* body0_b;  /* [64][4], [64]   */
  const float* body2_w; const float* body2_b;  /* [64][64], [64]  */
  const float* routing_w; const float* routing_b; /* [4][64], [4] */
  const float* offset_w; const float* offset_b;   /* [2][64], [2] */
  const float* st_offset_w; const float* st_offset_b;
  const float* compress; /* [4][8][64]  */
  const float* expand;   /* [4][64][8]  */
} savsr_satu_weights;

/*
 * Coordinate / index kernel (savsr_arch.py:326-351 and the grid of 262-288), fp32 with the exact
 * operation order of the reference (IEEE division, no FMA contraction):
 *   rel_y[H], rel_x[W]   R(.) = (q - floor(q + 1e-3)) - 0.5, q = (i + 0.5) / s
 *   cell_y[H], cell_x[W] int32 floor(q + 1e-3)              -- source LR cell
 *   base_y[H], base_x[W] fp32 normalised base grid coordinate (zero offset)
 *   corner_y[H], corner_x[W] int32 floor of the un-normalised base coordinate (may be -1)
 *   table [H*W][8] fp32 = (offset_x, offset_y, st_offset_x, st_offset_y, r0, r1, r2, r3) from the
 *   4->64->64 MLP and its three heads.  Depends only on (h, w, s_h, s_w): computed once per plan.
 * Any of the index outputs may be NULL.  H, W are passed in (python round() on the host, :745-751).
 */
int savsr_satu_index(savsr_ctx* ctx, const savsr_satu_weights* wts, int h, int w, int H, int W,
                     float s_h, float s_w, float* rel_y, float* rel_x, int32_t* cell_y,
                     int32_t* cell_x, float* base_y, float* base_x, int32_t* corner_y,
                     int32_t* corner_x, float* table, savsr_stream st);

/*
 * kernel_conv (1x1, 64 -> 64*25, LeakyReLU 0.1) and sta_conv (per-pixel 5x5 dynamic filtering, replicate padding on the
 * h x w region) of STAUpsample in ONE kernel (savsr_arch.py:297-313, 326): the 25 per-pixel kernels are produced tap by
 * tap on tcgen05 and consumed from TMEM, never written to memory.  a_slot: input of kernel_conv; x_slot: the feature
 * that is filtered; dst_slot: result.  weights: savsr_pack_conv_weight of the TAP-MAJOR filter [25*64][64][1][1]
 * (row t*64 + c = reference output channel c*25 + t), n_tile 64, SAVSR_ROWS_QUAD; bias fp32 [25][64] in the same order.
 */
int savsr_satu_kconv_sta(savsr_ctx* ctx, savsr_arena* arena, int a_slot, int x_slot, int dst_slot, int h, int w,
                         const void* weights, const float* bias, float slope, savsr_stream st);

/*
 * The whole HR side of SATU and the tail in ONE kernel, without any HR-resolution intermediate in memory
 * (savsr_arch.py:291 grid_sample x2, 353-370 routed compress / expand experts, 374 fusion, 738 tail conv, 739 bilinear skip):
 *   F = gather(x, offset), S = gather(sta, st_offset) ; U = F Wc^T ; V[e*8+k] = r_e sum_e' r_e' U[e'*8+k]
 *   Z[q][tap*3+c] = S[q] Wcs^T + F[q] Wcf^T + V[q] Wv^T + zbias       (fusion and tail composed on the host: both are linear)
 *   out[p][c] = tail_bias[c] + sum over the 3x3 taps inside the image of Z[p + d_tap][tap*3+c] + bilinear(x_center)[p][c]
 * weights: four [32 rows][128 B] K-major 128-byte-swizzled 16-bit tiles Wc | Wcf | Wcs | Wv (16 KB; rows of the last three =
 * tap*3+c, 27 used; Wv uses K = 32), in the context's format; zbias fp32 [32]; tail_bias fp32 [3];
 * x_in: the module's input window fp32 [batch][t][3][h][w]; out: fp32 NCHW [batch][3][H][W].
 * savsr_b200/engine.py (satu_hr_compose / satu_hr_pack) builds the operands from the reference's parameters.
 */
int savsr_satu_hr(savsr_ctx* ctx, savsr_arena* lr, int x_slot, int sta_slot, int h, int w, int H, int W,
                  const float* table, const float* base_y, const float* base_x, const void* weights,
                  const float* zbias, const float* tail_bias, const float* x_in, int t, int centre, float* out,
                  savsr_stream st);
/*
 * The same with 8-bit I/O: x_in is the uint8 BGR window [batch][t][h][w][3] given to savsr_pack_frames_u8 (the bilinear skip reads
 * its centre frame through the same u / 255), and out is uint8 HWC BGR [batch][H][W][3]: every pixel quantised as tensor2img does
 * (clamp to [0, 1], * 255, round half to even; what savsr_img_metrics writes to bgr_u8 from savsr_satu_hr's fp32 output).
 */
int savsr_satu_hr_u8(savsr_ctx* ctx, savsr_arena* lr, int x_slot, int sta_slot, int h, int w, int H, int W,
                     const float* table, const float* base_y, const float* base_x, const void* weights,
                     const float* zbias, const float* tail_bias, const uint8_t* x_in, int t, int centre, uint8_t* out,
                     savsr_stream st);
/* The same with the skip read from the frame table given to savsr_pack_frames_u8_table (entry n * t + centre); same ownership rule. */
int savsr_satu_hr_u8_table(savsr_ctx* ctx, savsr_arena* lr, int x_slot, int sta_slot, int h, int w, int H, int W,
                           const float* table, const float* base_y, const float* base_x, const void* weights,
                           const float* zbias, const float* tail_bias, const uint8_t* const* frames, int t, int centre, uint8_t* out,
                           savsr_stream st);
/* The same with 16-bit frames (savsr_pack_frames_u16_table): the skip reads the centre frame through v / 65535, and out is uint16 BGR
 * [batch][H][W][3], every pixel quantised as tensor2img does with 65535 in place of 255 (clamp to [0, 1], * 65535, round half to even). */
int savsr_satu_hr_u16_table(savsr_ctx* ctx, savsr_arena* lr, int x_slot, int sta_slot, int h, int w, int H, int W,
                            const float* table, const float* base_y, const float* base_x, const void* weights,
                            const float* zbias, const float* tail_bias, const uint16_t* const* frames, int t, int centre, uint16_t* out,
                            savsr_stream st);

/* ---- the forward as one call -----------------------------------------------------------------------------------------------------
 * savsr_plan = an ordered list of recorded launches of the entry points above (argument structures copied at record time), replayed on
 * a stream by savsr_plan_run; savsr_forward adds the copies between the caller's tensors and the plan's staging buffers
 * (SAVSR.forward, lbasicsr/archs/savsr_arch.py:692-742: x fp32 [batch][7][3][h][w] -> out fp32 [batch][3][H][W]).  A plan is built for one
 * (batch, h, w, scale) on buffers the caller prepared (arenas, packed weights, SATU tables: savsr_b200/engine.py does it); it owns no device
 * memory, never synchronises, and its replay is CUDA-graph capturable.  savsr_plan_add_* take the arguments of the corresponding
 * entry point minus the stream and return 0 / non-zero like everything else. */
typedef struct savsr_plan savsr_plan;
int savsr_plan_create(savsr_ctx* ctx, savsr_plan** out);
void savsr_plan_destroy(savsr_plan* plan);
int savsr_plan_size(const savsr_plan* plan);                 /* recorded launches */
int savsr_plan_set_io(savsr_plan* plan, float* x_in, size_t x_bytes, float* out, size_t out_bytes, int format /* enum savsr_format */);
/* 8-bit I/O: x_in uint8 BGR [batch][7][h][w][3], out uint8 BGR [batch][H][W][3] (the plan records savsr_pack_frames_u8 and
 * savsr_satu_hr_u8 on them).  A plan has one I/O mode, set by whichever of the two set_io calls came last. */
int savsr_plan_set_io_u8(savsr_plan* plan, uint8_t* x_in, size_t x_bytes, uint8_t* out, size_t out_bytes, int format);
/* 8-bit I/O from a frame table: table_dev is the device array of `entries` = batch * 7 frame pointers that the plan's
 * savsr_pack_frames_u8_table and savsr_satu_hr_u8_table launches read, out uint8 BGR [batch][H][W][3].  A third I/O mode. */
int savsr_plan_set_io_u8_table(savsr_plan* plan, const uint8_t** table_dev, int entries, uint8_t* out, size_t out_bytes, int format);
/* 16-bit I/O from a frame table of uint16 BGR frames (savsr_pack_frames_u16_table, savsr_satu_hr_u16_table), out uint16 BGR
 * [batch][H][W][3].  A fourth I/O mode. */
int savsr_plan_set_io_u16_table(savsr_plan* plan, const uint16_t** table_dev, int entries, uint16_t* out, size_t out_bytes, int format);
int savsr_plan_add_pack_frames(savsr_plan* plan, savsr_arena* arena, const float* x, int t, int h, int w, int dst_slot);
int savsr_plan_add_pack_frames_u8(savsr_plan* plan, savsr_arena* arena, const uint8_t* x, int t, int h, int w, int dst_slot);
int savsr_plan_add_pack_frames_u8_table(savsr_plan* plan, savsr_arena* arena, const uint8_t* const* frames, int t, int h, int w, int dst_slot);
int savsr_plan_add_pack_frames_u16_table(savsr_plan* plan, savsr_arena* arena, const uint16_t* const* frames, int t, int h, int w, int dst_slot);
int savsr_plan_add_conv(savsr_plan* plan, savsr_arena* arena, const savsr_conv_group* groups, int ngroups, int ksize, int n_tile,
                        int dst_mode, int impl);
int savsr_plan_add_osa_prologue(savsr_plan* plan, const savsr_osa_params* convs, int nconvs, int batch, int npart, int npix,
                                float inv_scale_h, float inv_scale_w);
int savsr_plan_add_ca_scale_residual(savsr_plan* plan, savsr_arena* arena, int t_slot, int x_slot, int dst_slot, const float* pool, int npart,
                                     const float* w1, const float* b1, const float* w2, const float* b2, float* y_scratch);
int savsr_plan_add_osadapt_mask(savsr_plan* plan, const float* in16, int batch, int height, int width, const float* wa, const float* ba,
                                const float* wb, const float* bb, const float* wc, const float* bc, float* half0, float* half1, float* mask);
int savsr_plan_add_satu_kconv_sta(savsr_plan* plan, savsr_arena* arena, int a_slot, int x_slot, int dst_slot, int h, int w, const void* weights,
                                  const float* bias, float slope);
int savsr_plan_add_satu_hr(savsr_plan* plan, savsr_arena* lr, int x_slot, int sta_slot, int h, int w, int H, int W, const float* table,
                           const float* base_y, const float* base_x, const void* weights, const float* zbias, const float* tail_bias,
                           const float* x_in, int t, int centre, float* out);
int savsr_plan_add_satu_hr_u8(savsr_plan* plan, savsr_arena* lr, int x_slot, int sta_slot, int h, int w, int H, int W, const float* table,
                              const float* base_y, const float* base_x, const void* weights, const float* zbias, const float* tail_bias,
                              const uint8_t* x_in, int t, int centre, uint8_t* out);
int savsr_plan_add_satu_hr_u8_table(savsr_plan* plan, savsr_arena* lr, int x_slot, int sta_slot, int h, int w, int H, int W, const float* table,
                                    const float* base_y, const float* base_x, const void* weights, const float* zbias, const float* tail_bias,
                                    const uint8_t* const* frames, int t, int centre, uint8_t* out);
int savsr_plan_add_satu_hr_u16_table(savsr_plan* plan, savsr_arena* lr, int x_slot, int sta_slot, int h, int w, int H, int W, const float* table,
                                     const float* base_y, const float* base_x, const void* weights, const float* zbias, const float* tail_bias,
                                     const uint16_t* const* frames, int t, int centre, uint16_t* out);
int savsr_plan_add_arena_export(savsr_plan* plan, savsr_arena* arena, int slot, float* nchw);   /* debug taps */
int savsr_plan_run(savsr_plan* plan, savsr_stream st);
/* x -> the plan's input staging buffer (device-to-device, skipped when x IS that buffer), replay, output staging buffer -> out. */
int savsr_forward(savsr_plan* plan, const float* x, float* out, savsr_stream st);
/* The same for a plan with 8-bit I/O (savsr_plan_set_io_u8): x uint8 BGR [batch][7][h][w][3] -> out uint8 BGR [batch][H][W][3].
 * Each of savsr_forward / savsr_forward_u8 returns an error, before any copy or launch, on a plan of the other I/O mode. */
int savsr_forward_u8(savsr_plan* plan, const uint8_t* x, uint8_t* out, savsr_stream st);
/* The same for a plan with frame-table I/O (savsr_plan_set_io_u8_table): ptrs_host holds batch * 7 DEVICE frame pointers, window n =
 * entries 7n .. 7n + 6, each one contiguous uint8 BGR [h][w][3] frame.  Writes the table (savsr_write_frame_table), replays, and copies
 * the output staging buffer to out uint8 BGR [batch][H][W][3].  The host array may be reused when the call returns; the frames must stay
 * valid, in stream order, until this forward has run.  Returns an error, before any launch, on a plan of another I/O mode, and
 * savsr_forward / savsr_forward_u8 refuse a frame-table plan. */
int savsr_forward_u8_frames(savsr_plan* plan, const uint8_t* const* ptrs_host, uint8_t* out, savsr_stream st);
/* The same for a plan with 16-bit frame-table I/O (savsr_plan_set_io_u16_table): each pointer is one contiguous uint16 BGR [h][w][3]
 * frame, out uint16 BGR [batch][H][W][3].  Same ownership rule; refuses a plan of another I/O mode before any launch, and the other
 * forward calls refuse this one. */
int savsr_forward_u16_frames(savsr_plan* plan, const uint16_t* const* ptrs_host, uint16_t* out, savsr_stream st);

/* ---- YUV 4:2:0 video in and out ------------------------------------------------------------------------------------------------
 * Decoders hand out and encoders take YUV 4:2:0, the forward reads and writes packed BGR.  These two calls convert on the device,
 * byte-identically to OpenCV's cv::cvtColor: COLOR_YUV2BGR_I420 / COLOR_YUV2BGR_NV12 (each pixel takes its 2x2 block's chroma sample)
 * and COLOR_BGR2YUV_I420 (U and V from the top-left pixel of each 2x2 block), with OpenCV's BT.601 limited-range matrix.  Video in another
 * matrix or range goes through the _cs calls below.  A C host decodes into a ring of BGR frames with savsr_yuv420_to_bgr, runs
 * savsr_forward_u8_frames on it, and encodes the output with savsr_bgr_to_yuv420.
 *
 * A YUV frame of h x w (both even) is described by its planes:
 *   y, y_pitch        the Y plane, h rows of w bytes, y_pitch >= w bytes apart;
 *   u, v, c_pitch     the chroma rows (h / 2 of them): chroma sample c of row r is u[r * c_pitch + c * c_step], likewise v;
 *   c_step            1 for yuv420p (I420: separate U and V planes of w / 2 bytes a row, c_pitch >= w / 2),
 *                     2 for nv12 (one plane of interleaved U, V bytes, U first: v = u + 1, c_pitch >= w);
 *   frame_stride      bytes from each plane of frame k to the same plane of frame k + 1.
 * ffmpeg's rawvideo yuv420p frame of [3h/2][w] bytes at p: y = p, y_pitch = w, u = p + h w, v = u + h w / 4, c_pitch = w / 2,
 * c_step = 1.  An NVDEC NV12 surface of pitch P at p: y = p, y_pitch = P, u = p + h P, v = u + 1, c_pitch = P, c_step = 2.
 * The BGR side is contiguous uint8 [n][h][w][3].  Both calls return an error before any launch on odd sizes, a null pointer, a pitch
 * below the row's width, a c_step other than 1 or 2, or a negative frame_stride; n = 0 launches nothing.
 * Ownership: every buffer must stay valid, in stream order, until the launch on st has run; the caller may reuse them after that.
 */
int savsr_yuv420_to_bgr(savsr_ctx* ctx, const uint8_t* y, int y_pitch, const uint8_t* u, const uint8_t* v, int c_pitch, int c_step,
                        int64_t frame_stride, int n, int h, int w, uint8_t* bgr, savsr_stream st);
int savsr_bgr_to_yuv420(savsr_ctx* ctx, const uint8_t* bgr, int n, int h, int w, uint8_t* y, int y_pitch, uint8_t* u, uint8_t* v,
                        int c_pitch, int c_step, int64_t frame_stride, savsr_stream st);
/*
 * 10-bit YUV 4:2:0 <-> 16-bit BGR (bgr48: contiguous uint16 [n][h][w][3], full scale 65535), for HEVC Main10 / 10-bit AV1 decoders and
 * encoders.  The same matrix and chroma handling as the two 8-bit calls, rescaled: one 10-bit step is a quarter of an 8-bit step, one
 * 8-bit BGR step is 257 sixteen-bit steps; decoding saturates to [0, 65535].  Each result is within 0.53 of an output step of the
 * real-valued map (fixed-point forms in savsr_b200/csrc/common.cuh).  The planes are described as above with every pitch and the
 * frame stride in uint16 elements, and
 *   msb = 0           yuv420p10le (ffmpeg): the value in bits 0-9; decoding reads s & 0x3ff, encoding writes the value;
 *   msb = 1           p010 (NVDEC 10-bit surfaces, c_step 2): the value in bits 6-15; decoding reads s >> 6, encoding writes v << 6.
 * A P010 surface of pitch P bytes at p: y = p, y_pitch = P / 2, u = y + h P / 2, v = u + 1, c_pitch = P / 2, c_step = 2, msb = 1.
 * Refusals as for the 8-bit calls, and an msb other than 0 or 1.
 */
int savsr_yuv420_10_to_bgr48(savsr_ctx* ctx, const uint16_t* y, int y_pitch, const uint16_t* u, const uint16_t* v, int c_pitch, int c_step,
                             int64_t frame_stride, int msb, int n, int h, int w, uint16_t* bgr, savsr_stream st);
int savsr_bgr48_to_yuv420_10(savsr_ctx* ctx, const uint16_t* bgr, int n, int h, int w, uint16_t* y, int y_pitch, uint16_t* u, uint16_t* v,
                             int c_pitch, int c_step, int64_t frame_stride, int msb, savsr_stream st);
/* ---- colour matrix and range (names as ffmpeg's -colorspace and -color_range) -------------------------------------------------------
 * The four conversions above for video in another matrix or range: each _cs call takes its plain call's arguments plus colorspace and
 * range.  (BT601, TV) launches exactly what the plain call launches (OpenCV's constants).  Every other pair converts with the
 * Y'CbCr <-> R'G'B' map of ITU-T H.273 (Kr, Kb: BT.601 0.299, 0.114; BT.709 0.2126, 0.0722; BT.2020 0.2627, 0.0593): tv range has
 * its black level at 16 and spans of 219 (Y) and 224 (U, V) 8-bit steps, pc range uses every code value (0 .. 2^n - 1, chroma
 * centred on 2^(n-1)).  Decoding rounds and saturates to [0, 255] or [0, 65535] without clamping Y at the black level; encoding rounds
 * and saturates to [0, 2^n - 1].  Integer forms within 0.55 of an output step of the real-valued map (savsr_b200/csrc/common.cuh).
 * Chroma handling, layouts, pitches and refusals are those of the plain calls; an unknown colorspace or range is refused, before any
 * launch, with a savsr_last_error() naming the value.  Only R'G'B' code values are produced: no transfer function (PQ, HLG) is applied,
 * and BT.2020 is the non-constant-luminance matrix.
 */
enum savsr_colorspace { SAVSR_COLORSPACE_BT601 = 0, SAVSR_COLORSPACE_BT709 = 1, SAVSR_COLORSPACE_BT2020NC = 2 };
enum savsr_color_range { SAVSR_RANGE_TV = 0, SAVSR_RANGE_PC = 1 };
int savsr_yuv420_to_bgr_cs(savsr_ctx* ctx, const uint8_t* y, int y_pitch, const uint8_t* u, const uint8_t* v, int c_pitch, int c_step,
                           int64_t frame_stride, int n, int h, int w, uint8_t* bgr, int colorspace, int range, savsr_stream st);
int savsr_bgr_to_yuv420_cs(savsr_ctx* ctx, const uint8_t* bgr, int n, int h, int w, uint8_t* y, int y_pitch, uint8_t* u, uint8_t* v,
                           int c_pitch, int c_step, int64_t frame_stride, int colorspace, int range, savsr_stream st);
int savsr_yuv420_10_to_bgr48_cs(savsr_ctx* ctx, const uint16_t* y, int y_pitch, const uint16_t* u, const uint16_t* v, int c_pitch,
                                int c_step, int64_t frame_stride, int msb, int n, int h, int w, uint16_t* bgr, int colorspace, int range,
                                savsr_stream st);
int savsr_bgr48_to_yuv420_10_cs(savsr_ctx* ctx, const uint16_t* bgr, int n, int h, int w, uint16_t* y, int y_pitch, uint16_t* u,
                                uint16_t* v, int c_pitch, int c_step, int64_t frame_stride, int msb, int colorspace, int range,
                                savsr_stream st);
/* ---- YUV 4:2:2 video in and out (mezzanine formats, capture devices) -----------------------------------------------------------
 * 4:2:2 halves the chroma horizontally only: frame row r has chroma row r, and each horizontal pixel pair shares one (U, V).  The
 * frame width must be even; any height is accepted.  Decoding gives both pixels of a pair its chroma (nearest neighbour: byte for byte
 * cv::cvtColor COLOR_YUV2BGR_YUYV / _UYVY at (BT601, TV)).  Encoding computes Y exactly as the 4:2:0 calls do and takes U and V from
 * the LEFT pixel of each pair: the co-sited chroma position of H.264, HEVC and ProRes 4:2:2 and the 4:2:0 calls' top-left rule, so a
 * 4:2:0 encode equals the 4:2:2 encode with its odd chroma rows dropped.  This is not COLOR_BGR2YUV_YUYV, which averages the pair's
 * chroma and rounds Y differently.  Every (colorspace, range) converts with the pixel map of the 4:2:0 calls: OpenCV's constants at
 * (BT601, TV), the H.273 map otherwise.  The planes are described as for 4:2:0, with chroma row r for frame row r, plus
 *   y_step            the distance between the Y samples of a row: 1 for the planar and semi-planar layouts, 2 for the packed ones;
 * and the layouts are
 *   yuv422p           y_step 1, c_step 1: Y plane, then U and V planes of h rows of w / 2 bytes (c_pitch >= w / 2); ffmpeg's [2h][w]
 *                     frame at p: y = p, y_pitch = w, u = p + h w, v = u + h w / 2, c_pitch = w / 2;
 *   nv16              y_step 1, c_step 2: Y plane, then h rows of interleaved U, V bytes, U first (v = u + 1, c_pitch >= w);
 *   yuyv422           y_step 2, c_step 4: rows of Y0 U0 Y1 V0 ...: u = y + 1, v = y + 3, c_pitch = y_pitch >= 2w;
 *   uyvy422           y_step 2, c_step 4: rows of U0 Y0 V0 Y1 ...: u = y - 1, v = y + 1, c_pitch = y_pitch >= 2w.
 * The 10-bit calls take yuv422p10le (c_step 1, msb 0) and p210 (c_step 2, msb 1: the value in bits 6-15, read as s >> 6, which also
 * reads 10-bit content in a P216 surface) with every pitch and the frame stride in uint16 elements, and bgr48 on the BGR side.
 * Refused before any launch, with a savsr_last_error() naming the value: an odd width, a (y_step, c_step) other than the layouts
 * above, a pitch below the row, a packed layout whose u and v are not those above, v != u + 1 for c_step 2, a null pointer, a negative
 * frame_stride, an msb other than 0 or 1, an unknown colorspace or range.  n = 0 launches nothing.  Ownership as for 4:2:0.
 */
int savsr_yuv422_to_bgr_cs(savsr_ctx* ctx, const uint8_t* y, int y_pitch, int y_step, const uint8_t* u, const uint8_t* v, int c_pitch,
                           int c_step, int64_t frame_stride, int n, int h, int w, uint8_t* bgr, int colorspace, int range, savsr_stream st);
int savsr_bgr_to_yuv422_cs(savsr_ctx* ctx, const uint8_t* bgr, int n, int h, int w, uint8_t* y, int y_pitch, int y_step, uint8_t* u,
                           uint8_t* v, int c_pitch, int c_step, int64_t frame_stride, int colorspace, int range, savsr_stream st);
int savsr_yuv422_10_to_bgr48_cs(savsr_ctx* ctx, const uint16_t* y, int y_pitch, int y_step, const uint16_t* u, const uint16_t* v,
                                int c_pitch, int c_step, int64_t frame_stride, int msb, int n, int h, int w, uint16_t* bgr, int colorspace,
                                int range, savsr_stream st);
int savsr_bgr48_to_yuv422_10_cs(savsr_ctx* ctx, const uint16_t* bgr, int n, int h, int w, uint16_t* y, int y_pitch, int y_step,
                                uint16_t* u, uint16_t* v, int c_pitch, int c_step, int64_t frame_stride, int msb, int colorspace, int range,
                                savsr_stream st);
/* uint8 BGR [n][h][w][3] -> uint16 BGR (each value times 257, so v / 65535 of the result is u / 255 of the source): brings 8-bit
 * frames into a ring of 16-bit frames, for an 8-bit source upscaled to deep output.  Both buffers contiguous; n = 0 launches nothing. */
int savsr_widen_u8_to_u16(savsr_ctx* ctx, const uint8_t* src, int n, int h, int w, uint16_t* dst, savsr_stream st);

/* ---- scene cuts in a streamed video ---------------------------------------------------------------------------------------------
 * A window that straddles a cut would mix two unrelated shots; instead each window is folded into its own shot, the reflection padding
 * the reference applies at the ends of a clip.  For the shot [start, stop) of frame c, L = stop - start, index i = c + o (o in -3 .. 3)
 * becomes start when L = 1, else start + r with r = (i - start) mod 2(L - 1) (non-negative), r replaced by 2(L - 1) - r when r >= L.
 * For L >= 4 this is the single reflection of a clip's ends.
 *
 * The caller keeps a ring of R >= 7 contiguous BGR [h][w][3] frames (frame t in slot t % R, as for savsr_forward_u8_frames) and three
 * small device arrays, sized by R alone: cut uint8 [R] and sad uint64 [R] (slot t % R belongs to frame t) and scratch uint64
 * [SAVSR_SCENE_SCRATCH_WORDS], zeroed once before the first call (each call leaves it ready for the next).  One detector state per ring.
 *
 * savsr_scene_score_u8 / _u16: after frame t has been written into its slot, scores it against frame t - 1:
 *   SAD_t = sum of |ring[t] - ring[t - 1]| over all 3hw samples (SAD_0 = 0),   m_t = min(SAD_t, |SAD_t - SAD_{t-1}|)
 * (ffmpeg scdet's min(mafd, |mafd - prev_mafd|), scaled), and writes sad[t % R] = SAD_t and cut[t % R] = 1 when t >= 1 and
 * m_t >= bound, or when `marked` (a cut the caller knows of, e.g. from an edit list), else 0.  For a threshold tau in percent, the
 * score 100 m_t / (3hw maxval) reaches tau exactly when m_t >= bound = ceil(tau * 3hw * maxval / 100), maxval 255 or 65535, which the
 * host computes from the exact value of tau.
 * Because maxval is the full scale, an 8-bit source widened by 257 gets the decisions of the 8-bit frames.  A cut that ends a 1-frame
 * shot is not detected: its SAD and the one before it cancel in |SAD_t - SAD_{t-1}|, as scdet suppresses a flash; mark such cuts.
 * Call once per frame, t = 0, 1, 2, ... in order on one stream (frame t reads sad[(t - 1) % R] written by the call of t - 1); t = 0
 * starts a new video.  One launch, integer arithmetic: the result does not depend on the launch configuration.
 *
 * savsr_write_scene_frame_table: writes the 7 * count table entries of the windows of frames first .. first + count - 1, each folded into
 * its shot, where a shot starts at frame 0 and at every frame whose cut flag is set: entry 7n + k = ring + ((window entry k of frame
 * first + n) % R) * frame_bytes.  `received` frames have been scored so far; `finished` = 1 once the stream has ended (the last shot
 * ends at `received`), else every window must lie inside the received frames (first + count + 2 < received).  It reads only the flags
 * of frames c - 2 .. c + 3 of each window, never a frame not yet received, so the host needs no read-back of the flags.
 *
 * Composition on one stream (what savsr_b200.VideoUpscaler does with a plan of savsr_plan_set_io_u8_table / _u16_table): per frame t,
 * write it into slot t % R and call savsr_scene_score; when frame j + 2 has arrived (or at the end), call savsr_write_scene_frame_table
 * with the plan's table and count = the plan's batch, then savsr_plan_run (or a graph replay of it), then read the plan's output.  The
 * table writer replaces savsr_write_frame_table and runs, like it, in stream order outside any captured graph.
 * Ownership: the ring, the arrays and the table must stay valid, in stream order, until the launches that read them have run; a ring slot
 * may be rewritten only after every launch that reads it was enqueued.  Both calls return an error before any launch on a null pointer,
 * R < 7, a non-positive bound or frame size, and (the writer) a batch that reaches past the received frames or beyond the ring.
 */
#define SAVSR_SCENE_SCRATCH_WORDS 1024
int savsr_scene_score_u8(savsr_ctx* ctx, const uint8_t* ring, int R, int h, int w, long long t, int marked, long long bound, uint8_t* cut,
                         unsigned long long* sad, unsigned long long* scratch, savsr_stream st);
int savsr_scene_score_u16(savsr_ctx* ctx, const uint16_t* ring, int R, int h, int w, long long t, int marked, long long bound, uint8_t* cut,
                          unsigned long long* sad, unsigned long long* scratch, savsr_stream st);
int savsr_write_scene_frame_table(savsr_ctx* ctx, const uint8_t** table_dev, const void* ring, long long frame_bytes, int R, const uint8_t* cut,
                                  long long first, int count, long long received, int finished, savsr_stream st);

/* ---- post-processing / metrics on the device (next row 8f3) -------------------------------------------------------
 * tensor2img (lbasicsr/utils/img_util.py:38-94): sr fp32 NCHW [batch][3][H][W] RGB -> uint8 HWC BGR [batch][H][W][3]
 * (clamp, *255, round half to even), and, when gt is given, the per-frame sum of squared Y-channel differences of the two
 * uint8 images (metric_util.py:32-45, color_util.py:38-68, psnr_ssim.py:11-48 with crop_border 0) in float64, as one partial
 * sum per thread block: sse_y [batch][savsr_img_metrics_blocks(ctx, H, W)], SSE_n = sum(sse_y[n]) in a fixed order (bit-reproducible),
 * PSNR_Y = 10 log10(255^2 * H*W / SSE_n).  bgr_u8 and sse_y may each be NULL.
 */
int savsr_img_metrics_blocks(const savsr_ctx* ctx, int height, int width);
int savsr_img_metrics(savsr_ctx* ctx, const float* sr, const float* gt, int batch, int height, int width,
                      uint8_t* bgr_u8, double* sse_y, savsr_stream st);

/*
 * SSIM on the Y channel of the same uint8 images (lbasicsr/metrics/psnr_ssim.py:85-129 and _ssim 172-200 with
 * crop_border 0, test_y_channel true; the YAML metric `ssim_y`): 11x11 Gaussian window (sigma 1.5), fully covered
 * positions only, float64.  Writes one partial sum per 16x16 block of the SSIM map:
 * partials [batch][savsr_ssim_y_blocks(H, W)], SSIM_n = sum(partials[n]) / ((H - 10) * (W - 10)).  Needs H, W >= 11.
 */
int savsr_ssim_y_blocks(int height, int width);
int savsr_ssim_y(savsr_ctx* ctx, const float* sr, const float* gt, int batch, int height, int width,
                 double* partials, savsr_stream st);

/* ---- LR synthesis on the device (next row 8f2) ------------------------------------------------------------------------
 * The reference builds every LR window on the CPU from the uint8 ground-truth frames
 * (lbasicsr/data/video_test_dataset.py:297-328): cv2.imread / 255 (data_util.py:41) -> as_mod_crop (transforms.py:47-69)
 * -> img2tensor (BGR->RGB, CHW) -> torchvision Resize(size, BICUBIC, antialias=True) (data_util.py:396-412), i.e. ATen's
 * _upsample_bicubic2d_aa.  These entry points do the same on frames resident in HBM, bit-exactly (width pass first into a
 * float32 intermediate, a = -0.5 bicubic taps normalised in float32, the accumulation order of the ATen CPU kernel).
 *
 * savsr_aa_max_taps: row stride the caller must give the weight table of one axis.
 * savsr_aa_table:    per output index, first source index, tap count and weights [out_size][max_taps]; *overflow_flag
 *                    (device int) is set to 1 if a row needed more than max_taps taps (cannot happen with the size above).
 * savsr_lr_synthesize: frames_bgr uint8 [n][H][W][3] -> lr fp32 [n][3][out_h][out_w] (tmp: [n][3][crop_h][out_w] scratch)
 *                    and, if gt != NULL, the mod-cropped ground truth fp32 RGB [n][3][crop_h][crop_w].  The crop is the
 *                    top-left crop_h x crop_w region (as_mod_crop); an axis whose size does not change needs no table.
 */
int savsr_aa_max_taps(int in_size, int out_size);
int savsr_aa_table(savsr_ctx* ctx, int in_size, int out_size, int max_taps, int32_t* xmin, int32_t* xsize,
                   float* weights, int32_t* overflow_flag, savsr_stream st);
int savsr_lr_synthesize(savsr_ctx* ctx, const uint8_t* frames_bgr, int nframes, int height, int width,
                        int crop_h, int crop_w, int out_h, int out_w,
                        const int32_t* xmin_w, const int32_t* xsize_w, const float* weights_w, int taps_w,
                        const int32_t* xmin_h, const int32_t* xsize_h, const float* weights_h, int taps_h,
                        float* tmp, float* lr, float* gt, savsr_stream st);
/*
 * Row 8f4: the reference resizes an SR result whose size differs from the ground truth with the same antialiased bicubic
 * Resize before the metrics (lbasicsr/models/sr_model.py:291-304).  src fp32 [n][3][H][W] -> dst fp32 [n][3][out_h][out_w]
 * (tmp: [n][3][H][out_w] scratch), tables from savsr_aa_table; same separable float32 arithmetic as savsr_lr_synthesize.
 */
int savsr_resize_aa(savsr_ctx* ctx, const float* src, int nframes, int height, int width, int out_h, int out_w,
                    const int32_t* xmin_w, const int32_t* xsize_w, const float* weights_w, int taps_w,
                    const int32_t* xmin_h, const int32_t* xsize_h, const float* weights_h, int taps_h,
                    float* tmp, float* dst, savsr_stream st);

#ifdef __cplusplus
}
#endif
#endif /* SAVSR_B200_H_ */
