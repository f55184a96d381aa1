// Shared device helpers for libsavsr_sm100: PTX wrappers for mbarrier / TMA / tcgen05 (sm_100a only),
// bf16 packing, error plumbing.  Hand-written; no CUTLASS dependency.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/savsr_b200.h"

namespace savsr {

// ------------------------------------------------------------------------------------------------ host side
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define SAVSR_CUDA(expr)                                   \
  do {                                                     \
    cudaError_t _e = (expr);                               \
    if (_e != cudaSuccess) return ::savsr::cuda_fail(_e, #expr); \
  } while (0)

#define SAVSR_REQUIRE(cond, ...)          \
  do {                                    \
    if (!(cond)) {                        \
      ::savsr::set_error(__VA_ARGS__);    \
      return 1;                           \
    }                                     \
  } while (0)

constexpr int kTileW = SAVSR_TILE_W;
constexpr int kTileH = SAVSR_TILE_H;
constexpr int kTileM = kTileW * kTileH;  // 128
constexpr int kC = 64;                   // channels per arena slot

}  // namespace savsr

struct savsr_ctx {
  int device;
  int sm_count;
  int cc_major, cc_minor;
  void* encode_tiled;  // PFN_cuTensorMapEncodeTiled
  int fmt;             // 16-bit storage / operand format of arenas and packed weights: SAVSR_FMT_BF16 or SAVSR_FMT_FP16
  int opt[SAVSR_OPT_COUNT];   // enum savsr_option values (savsr_ctx_set_option)
  uint32_t attr_mask;  // bit k: the dynamic shared-memory attribute of kernel k is set on THIS context's device
  long long* conv_dbg; // SAVSR_DEBUG_COUNTERS builds only: device buffer [grid][8] for cycle counters, else unused
};

namespace savsr {
// Kernels that need more than 48 KB of dynamic shared memory: the attribute belongs to the device (primary context), so
// it is tracked per savsr_ctx, not per process.
enum AttrBit { kAttrIgemm = 0 /* + template index, 6 variants */, kAttrBigk = 8, kAttrKsta = 9, kAttrSatuHr = 10, kAttrOsaLinear = 11,
               kAttrFused = 12, kAttrBigk128 = 13, kAttrSatuHrBf16 = 14, kAttrWgrad = 15, kAttrWgradBatched = 16,
               kAttrOsaAssembleTrain = 17, kAttrOsaUnfoldBwd = 18, kAttrOsaChain = 19, kAttrOsaMatvec = 20 /* + 0, 1, 2: batch 8, 16, 32 */,
               kAttrCaBackward = 23, kAttrSatuHrU8 = 24 /* + format: 8-bit I/O instantiations of satu_hr */ };
template <class F>
inline int ensure_smem_attr(savsr_ctx* ctx, int bit, F func, size_t bytes) {
  if (ctx->attr_mask & (1u << bit)) return 0;
  SAVSR_CUDA(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes)));
  ctx->attr_mask |= 1u << bit;
  return 0;
}
// Kernel launch with optional programmatic dependent launch (SAVSR_OPT_PDL): the kernel must call pdl_wait() before its first access to
// memory a previous kernel may have written, and may call pdl_trigger() after it.
template <class... KArgs, class... Args>
inline cudaError_t launch_k(bool pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
// Launch on the context's device whatever the caller's current device is; restores it on scope exit.  cudaSetDevice is called
// even when the device already matches: it also binds the primary context to the calling THREAD, which a fresh thread (e.g.
// autograd's backward worker) does not have yet -- the driver entry points (cuTensorMapEncodeTiled) fail with
// CUDA_ERROR_INVALID_CONTEXT otherwise.
struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  explicit DeviceGuard(int device) {
    const bool known = cudaGetDevice(&prev) == cudaSuccess;
    const bool ok = cudaSetDevice(device) == cudaSuccess;
    switched = known && ok && prev != device;
  }
  ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
};
}  // namespace savsr

struct savsr_arena {
  savsr_ctx* ctx;
  __nv_bfloat16* base;
  int nslots, batch, height, width;
  int tiles_x, tiles_y;
  CUtensorMap tm_tile;  // box [64, 8, 16, 1]
  CUtensorMap tm_halo;  // box [64, 10, 18, 1]
};

#ifdef __CUDACC__
namespace savsr {

// ------------------------------------------------------------------------------------------------ misc
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// Two 16-bit floats <-> fp32.  fmt = SAVSR_FMT_BF16 (0) or SAVSR_FMT_FP16 (1); warp-uniform, so the select is free.
__device__ __forceinline__ uint32_t pack_h2(float lo, float hi, int fmt) {
  if (fmt) {
    __half2 v = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
  }
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float h_lo(uint32_t v, int fmt) {
  return fmt ? __half2float(__ushort_as_half(static_cast<unsigned short>(v & 0xffffu))) : __uint_as_float(v << 16);
}
__device__ __forceinline__ float h_hi(uint32_t v, int fmt) {
  return fmt ? __half2float(__ushort_as_half(static_cast<unsigned short>(v >> 16))) : __uint_as_float(v & 0xffff0000u);
}
// 8-bit pixel <-> [0, 1] float.  In: the reference's img.astype(np.float32) / 255., correctly rounded.  A multiply by the rounded
// reciprocal alone is off by one ulp for 126 of the 256 values; with one fma correction of the remainder it is exact for all of them
// (checked exhaustively, tests/test_video_u8_io.py), and unlike __fdiv_rn it has no slow-path call.
// Out: tensor2img (lbasicsr/utils/img_util.py:38-94): clamp to [0, 1], * 255, round half to even.
__device__ __forceinline__ float u8_to_unit(uint8_t u) {
  const float a = static_cast<float>(u), r = 1.0f / 255.0f;
  const float q = __fmul_rn(a, r);
  return __fmaf_rn(__fmaf_rn(-q, 255.0f, a), r, q);
}
__device__ __forceinline__ int unit_to_u8(float v) { return __float2int_rn(fminf(fmaxf(v, 0.f), 1.f) * 255.0f); }
__device__ __forceinline__ float h_to_float(uint16_t raw, int fmt) { return h_lo(raw, fmt); }
__device__ __forceinline__ uint16_t float_to_h(float x, int fmt) { return static_cast<uint16_t>(pack_h2(x, 0.f, fmt) & 0xffffu); }

// ATen upsample_bilinear2d, align_corners = False (savsr_arch.py:739): source index and weight.
__device__ __forceinline__ void bilinear_src(int dst, int in_size, int out_size, int& i0, int& i1, float& l1) {
  const float scale = static_cast<float>(in_size) / static_cast<float>(out_size);
  float src = scale * (static_cast<float>(dst) + 0.5f) - 0.5f;
  src = src < 0.f ? 0.f : src;
  i0 = static_cast<int>(src);
  i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
  l1 = src - static_cast<float>(i0);
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// Named barrier over a subset of the CTA's warps (id 1..15; `count` = participating threads, multiple of 32).
__device__ __forceinline__ void named_barrier(int id, int count) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// Programmatic dependent launch: block until the preceding kernel of the stream has completed and its writes are visible (a no-op when
// the kernel was launched normally); then allow the next kernel's CTAs to be scheduled as this grid's CTAs retire.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Spin with a bounded trip count: a protocol bug traps instead of hanging the GPU box.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) {
      printf("savsr: mbarrier timeout block %d thread %d bar %p parity %u\n", blockIdx.x, threadIdx.x,
             (void*)bar, parity);
      __trap();
    }
  }
}

// ------------------------------------------------------------------------------------------------ TMA
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}
// 4-D tiled load: coordinates (c, x, y, img), out-of-range elements are zero-filled.
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* tm, uint64_t* bar, int c, int x,
                                            int y, int img) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%2, %3, %4, %5}], [%6];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c), "r"(x), "r"(y), "r"(img),
      "r"(smem_u32(bar))
      : "memory");
}
// Same box, fetched into L2 only (no shared-memory destination, no completion signal): hides DRAM latency for a later
// tma_load_4d of the same coordinates without holding a pipeline stage.
__device__ __forceinline__ void tma_prefetch_4d(const CUtensorMap* tm, int c, int x, int y, int img) {
  asm volatile("cp.async.bulk.prefetch.tensor.4d.L2.global.tile [%0, {%1, %2, %3, %4}];"
               ::"l"(reinterpret_cast<uint64_t>(tm)), "r"(c), "r"(x), "r"(y), "r"(img)
               : "memory");
}
// 1-D bulk copy global -> shared (size multiple of 16 bytes, both 16-byte aligned).
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ------------------------------------------------------------------------------------------------ tcgen05
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

template <int kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_out) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_out)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {  // same warp that allocated
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}

// Shared-memory matrix descriptor, K-major operand, 128-byte swizzle (layout_type 2), version 1.
//   start address >> 4 in bits [0,14); LBO unused for a single swizzle atom along K;
//   SBO (bytes between 8-row groups) >> 4 in bits [32,46); base_offset in bits [49,52).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr, uint32_t sbo_bytes, uint32_t base_offset) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr >> 4) & 0x3fffu);
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3fffu) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(base_offset & 7u) << 49;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

// Instruction descriptor for kind::f16: (bf16 | fp16) x same -> fp32, both operands K-major, M = 128.
__host__ __device__ constexpr uint32_t umma_idesc_f16(int n, int fmt) {
  return (1u << 4)                              // c_format  = F32
         | ((fmt ? 0u : 1u) << 7)               // a_format  = BF16 (1) / F16 (0)
         | ((fmt ? 0u : 1u) << 10)              // b_format
         | (static_cast<uint32_t>(n >> 3) << 17)  // N >> 3
         | (static_cast<uint32_t>(128 >> 4) << 24);  // M >> 4
}

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// SAVSR_ROWS_QUAD row order of a packed N = 64 weight block: row (= accumulator column) n holds output channel
// quad_row(n), the bit fields [2:1] and [4:3] of n swapped.  With it the 8 accumulator columns one thread receives from
// a 16x256b.x4 TMEM load (8 k + 2 q + e) are the 8 CONSECUTIVE channels 8 q + 2 k + e, so conv epilogues read and write
// 16 contiguous bytes per thread and 64 per thread quad without any transposition.  The map is its own inverse.
__host__ __device__ __forceinline__ int quad_row(int n) { return (n & 0x21) | (((n >> 1) & 3) << 3) | (((n >> 3) & 3) << 1); }

// 32 lanes x 32 bit, 16 consecutive columns: thread i of the warp gets TMEM lane (base_lane + i).
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 16 lanes x 256 bit, repeated 4 times along the columns (32 columns): thread t = 4 g + q of the warp receives
//   v[4 k + e] = TMEM[lane base + g + 8 (e >> 1)][column base + 8 k + 2 q + (e & 1)],  k = 0..3, e = 0..3
// (the mma.sync accumulator-fragment layout; measured with scripts/tmem_layout.cu).  The address' lane field selects
// the first of the 16 lanes, so a warp covers its 32-lane quadrant with two loads (lane offsets 0 and 16).
__device__ __forceinline__ void tmem_ld_16x256b_x4(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}

}  // namespace savsr
#endif  // __CUDACC__
