// LR synthesis on the device (SURVEY.md section 8 row f2): uint8 BGR ground-truth frames -> float32 RGB, arbitrary-scale
// mod crop, antialiased bicubic downsample.  Replaces, per output frame, the CPU chain of the reference
//   cv2.imread / 255 (lbasicsr/data/data_util.py:41) -> as_mod_crop (transforms.py:47-69) -> img2tensor ->
//   T.Resize(size, BICUBIC, antialias=True) (data_util.py:396-412)
// and is bit-exact with it: the resampling follows ATen's _upsample_bicubic2d_aa CPU kernel operation by operation,
// including the fused multiply-adds its x86-64 build contains (see oracle/lr_synthesis.py for the derivation).  All
// arithmetic that must round like the reference uses explicit __f*_rn / __d*_rn intrinsics so nvcc cannot re-associate
// or contract it differently.
#include <math.h>

#include "common.cuh"

namespace savsr {

__device__ __forceinline__ float aa_cubic(float x) {
  if (x < 1.0f) {
    float t = __fmaf_rn(1.5f, x, -2.5f);
    t = __fmul_rn(t, x);
    return __fmaf_rn(t, x, 1.0f);
  }
  if (x < 2.0f) {
    float t = __fmaf_rn(-0.5f, x, 2.5f);
    t = __fmaf_rn(t, x, -4.0f);
    return __fmaf_rn(t, x, 2.0f);
  }
  return 0.0f;
}

// One thread per output index: xmin, xsize and the normalised weights (row stride max_taps).
__global__ void aa_table_kernel(int in_size, int out_size, int max_taps, int32_t* __restrict__ xmin_out,
                                int32_t* __restrict__ xsize_out, float* __restrict__ weights, int* __restrict__ overflow) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= out_size) return;
  const float scale = __fdiv_rn(static_cast<float>(in_size), static_cast<float>(out_size));
  const float support = scale >= 1.0f ? __fmul_rn(2.0f, scale) : 2.0f;
  const float invscale = scale >= 1.0f ? static_cast<float>(__ddiv_rn(1.0, static_cast<double>(scale))) : 1.0f;
  const float center = static_cast<float>(__dmul_rn(static_cast<double>(scale), static_cast<double>(i) + 0.5));
  int xmin = static_cast<int>(__dadd_rn(static_cast<double>(__fsub_rn(center, support)), 0.5));   // truncation, like the C cast
  xmin = xmin > 0 ? xmin : 0;
  int xend = static_cast<int>(__dadd_rn(static_cast<double>(__fadd_rn(center, support)), 0.5));
  xend = xend < in_size ? xend : in_size;
  int xsize = xend - xmin;
  if (xsize > max_taps) { atomicExch(overflow, 1); xsize = max_taps; }
  float* w = weights + static_cast<long>(i) * max_taps;
  float total = 0.0f;
  for (int j = 0; j < xsize; ++j) {
    const double d = __dadd_rn(static_cast<double>(__fsub_rn(static_cast<float>(j + xmin), center)), 0.5);
    const float x = fabsf(static_cast<float>(__dmul_rn(d, static_cast<double>(invscale))));
    const float v = aa_cubic(x);
    w[j] = v;
    total = __fadd_rn(total, v);
  }
  if (total != 0.0f) {
    for (int j = 0; j < xsize; ++j) w[j] = __fdiv_rn(w[j], total);
  }
  for (int j = xsize; j < max_taps; ++j) w[j] = 0.0f;
  xmin_out[i] = xmin;
  xsize_out[i] = xsize;
}

// t = s[0] w[0]; t += s[j] w[j]: 4-way unrolled multiply + add main loop, fused remainder (ATen 2.11.0 x86-64 build).
template <class Load>
__device__ __forceinline__ float aa_accumulate(Load load, const float* __restrict__ w, int n) {
  float t = __fmul_rn(load(0), w[0]);
  const int main_end = ((n - 1) >> 2) << 2;
  for (int j = 1; j <= main_end; ++j) t = __fadd_rn(t, __fmul_rn(load(j), w[j]));
  for (int j = main_end + 1; j < n; ++j) t = __fmaf_rn(load(j), w[j], t);
  return t;
}

struct LrParams {
  const uint8_t* frames;   // [n][H][W][3] BGR, or nullptr when `planes` is the source
  const float* planes;     // [n][3][H][W] float32 (post-resize of SR frames, row f4), top-left hc x wc region used
  int n, H, W, hc, wc, oh, ow;
  const int32_t *xmin_w, *xsize_w, *xmin_h, *xsize_h;
  const float *wt_w, *wt_h;
  int taps_w, taps_h;
  float* tmp;   // [n][3][hc][ow]
  float* lr;    // [n][3][oh][ow]
  float* gt;    // [n][3][hc][wc] or nullptr
};

// width pass straight from the uint8 frames (x / 255 and BGR -> RGB fused); identity when the width does not change
__global__ void __launch_bounds__(256) lr_width_kernel(const LrParams p) {
  const long total = static_cast<long>(p.n) * 3 * p.hc * p.ow;
  for (long idx = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; idx < total; idx += static_cast<long>(gridDim.x) * blockDim.x) {
    const int ox = idx % p.ow;
    long r = idx / p.ow;
    const int y = r % p.hc; r /= p.hc;
    const int c = r % 3;
    const int t = r / 3;
    float v;
    if (p.frames != nullptr) {
      const uint8_t* row = p.frames + ((static_cast<long>(t) * p.H + y) * p.W) * 3 + (2 - c);
      auto load = [&](int x) { return u8_to_unit(row[static_cast<long>(x) * 3]); };
      if (p.ow == p.wc) {
        v = load(ox);
      } else {
        const int x0 = p.xmin_w[ox];
        v = aa_accumulate([&](int j) { return load(x0 + j); }, p.wt_w + static_cast<long>(ox) * p.taps_w, p.xsize_w[ox]);
      }
    } else {
      const float* row = p.planes + ((static_cast<long>(t) * 3 + c) * p.H + y) * p.W;
      if (p.ow == p.wc) {
        v = row[ox];
      } else {
        const int x0 = p.xmin_w[ox];
        v = aa_accumulate([&](int j) { return row[x0 + j]; }, p.wt_w + static_cast<long>(ox) * p.taps_w, p.xsize_w[ox]);
      }
    }
    p.tmp[idx] = v;
  }
}

// height pass on the float32 intermediate; identity when the height does not change
__global__ void __launch_bounds__(256) lr_height_kernel(const LrParams p) {
  const long total = static_cast<long>(p.n) * 3 * p.oh * p.ow;
  for (long idx = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; idx < total; idx += static_cast<long>(gridDim.x) * blockDim.x) {
    const int ox = idx % p.ow;
    long r = idx / p.ow;
    const int oy = r % p.oh;
    const long tc = r / p.oh;
    const float* col = p.tmp + tc * p.hc * p.ow + ox;
    float v;
    if (p.oh == p.hc) {
      v = col[static_cast<long>(oy) * p.ow];
    } else {
      const int y0 = p.xmin_h[oy];
      v = aa_accumulate([&](int j) { return col[static_cast<long>(y0 + j) * p.ow]; }, p.wt_h + static_cast<long>(oy) * p.taps_h, p.xsize_h[oy]);
    }
    p.lr[idx] = v;
  }
}

// mod-cropped ground truth as float32 RGB CHW (what the reference hands to the metrics)
__global__ void __launch_bounds__(256) gt_rgb_kernel(const LrParams p) {
  const long total = static_cast<long>(p.n) * 3 * p.hc * p.wc;
  for (long idx = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; idx < total; idx += static_cast<long>(gridDim.x) * blockDim.x) {
    const int x = idx % p.wc;
    long r = idx / p.wc;
    const int y = r % p.hc; r /= p.hc;
    const int c = r % 3;
    const int t = r / 3;
    p.gt[idx] = u8_to_unit(p.frames[((static_cast<long>(t) * p.H + y) * p.W + x) * 3 + (2 - c)]);
  }
}

}  // namespace savsr

using namespace savsr;

extern "C" int savsr_aa_max_taps(int in_size, int out_size) {
  if (in_size <= 0 || out_size <= 0) return 0;
  const float scale = static_cast<float>(in_size) / static_cast<float>(out_size);
  const float support = scale >= 1.0f ? 2.0f * scale : 2.0f;
  return static_cast<int>(ceilf(2.0f * support)) + 2;
}

extern "C" int savsr_aa_table(savsr_ctx* ctx, int in_size, int out_size, int max_taps, int32_t* xmin, int32_t* xsize,
                              float* weights, int32_t* overflow_flag, savsr_stream st) {
  SAVSR_REQUIRE(ctx && xmin && xsize && weights && overflow_flag, "savsr_aa_table: null pointer");
  DeviceGuard guard(ctx->device);
  SAVSR_REQUIRE(in_size > 0 && out_size > 0, "savsr_aa_table: sizes must be positive (%d -> %d)", in_size, out_size);
  SAVSR_REQUIRE(max_taps >= savsr_aa_max_taps(in_size, out_size), "savsr_aa_table: max_taps %d < savsr_aa_max_taps = %d", max_taps,
                savsr_aa_max_taps(in_size, out_size));
  SAVSR_CUDA(cudaMemsetAsync(overflow_flag, 0, sizeof(int32_t), static_cast<cudaStream_t>(st)));
  aa_table_kernel<<<(out_size + 127) / 128, 128, 0, static_cast<cudaStream_t>(st)>>>(in_size, out_size, max_taps, xmin, xsize, weights,
                                                                                    overflow_flag);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int savsr_lr_synthesize(savsr_ctx* ctx, const uint8_t* frames_bgr, int nframes, int height, int width, int crop_h,
                                   int crop_w, int out_h, int out_w, const int32_t* xmin_w, const int32_t* xsize_w,
                                   const float* weights_w, int taps_w, const int32_t* xmin_h, const int32_t* xsize_h,
                                   const float* weights_h, int taps_h, float* tmp, float* lr, float* gt, savsr_stream st_) {
  SAVSR_REQUIRE(ctx && frames_bgr && tmp && lr, "savsr_lr_synthesize: null pointer");
  DeviceGuard guard(ctx->device);
  SAVSR_REQUIRE(nframes >= 0 && height > 0 && width > 0, "savsr_lr_synthesize: bad frame shape");
  SAVSR_REQUIRE(crop_h > 0 && crop_h <= height && crop_w > 0 && crop_w <= width, "savsr_lr_synthesize: crop %dx%d outside the %dx%d frame",
                crop_h, crop_w, height, width);
  SAVSR_REQUIRE(out_h > 0 && out_w > 0, "savsr_lr_synthesize: bad output size %dx%d", out_h, out_w);
  SAVSR_REQUIRE(out_w == crop_w || (xmin_w && xsize_w && weights_w && taps_w > 0), "savsr_lr_synthesize: width tables missing");
  SAVSR_REQUIRE(out_h == crop_h || (xmin_h && xsize_h && weights_h && taps_h > 0), "savsr_lr_synthesize: height tables missing");
  if (nframes == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(st_);
  LrParams p;
  p.frames = frames_bgr; p.planes = nullptr; p.n = nframes; p.H = height; p.W = width; p.hc = crop_h; p.wc = crop_w; p.oh = out_h; p.ow = out_w;
  p.xmin_w = xmin_w; p.xsize_w = xsize_w; p.wt_w = weights_w; p.taps_w = taps_w;
  p.xmin_h = xmin_h; p.xsize_h = xsize_h; p.wt_h = weights_h; p.taps_h = taps_h;
  p.tmp = tmp; p.lr = lr; p.gt = gt;
  auto blocks = [&](long total) {
    long b = (total + 255) / 256;
    const long cap = 16L * ctx->sm_count;
    return static_cast<unsigned>(b < cap ? b : cap);
  };
  lr_width_kernel<<<blocks(static_cast<long>(nframes) * 3 * crop_h * out_w), 256, 0, st>>>(p);
  lr_height_kernel<<<blocks(static_cast<long>(nframes) * 3 * out_h * out_w), 256, 0, st>>>(p);
  if (gt != nullptr) gt_rgb_kernel<<<blocks(static_cast<long>(nframes) * 3 * crop_h * crop_w), 256, 0, st>>>(p);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int savsr_resize_aa(savsr_ctx* ctx, const float* src, int nframes, int height, int width, int out_h, int out_w,
                               const int32_t* xmin_w, const int32_t* xsize_w, const float* weights_w, int taps_w,
                               const int32_t* xmin_h, const int32_t* xsize_h, const float* weights_h, int taps_h, float* tmp,
                               float* dst, savsr_stream st_) {
  SAVSR_REQUIRE(ctx && src && tmp && dst, "savsr_resize_aa: null pointer");
  DeviceGuard guard(ctx->device);
  SAVSR_REQUIRE(nframes >= 0 && height > 0 && width > 0 && out_h > 0 && out_w > 0, "savsr_resize_aa: bad shape");
  SAVSR_REQUIRE(out_w == width || (xmin_w && xsize_w && weights_w && taps_w > 0), "savsr_resize_aa: width tables missing");
  SAVSR_REQUIRE(out_h == height || (xmin_h && xsize_h && weights_h && taps_h > 0), "savsr_resize_aa: height tables missing");
  if (nframes == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(st_);
  LrParams p;
  p.frames = nullptr; p.planes = src; p.n = nframes; p.H = height; p.W = width; p.hc = height; p.wc = width; p.oh = out_h; p.ow = out_w;
  p.xmin_w = xmin_w; p.xsize_w = xsize_w; p.wt_w = weights_w; p.taps_w = taps_w;
  p.xmin_h = xmin_h; p.xsize_h = xsize_h; p.wt_h = weights_h; p.taps_h = taps_h;
  p.tmp = tmp; p.lr = dst; p.gt = nullptr;
  auto blocks = [&](long total) {
    long b = (total + 255) / 256;
    const long cap = 16L * ctx->sm_count;
    return static_cast<unsigned>(b < cap ? b : cap);
  };
  lr_width_kernel<<<blocks(static_cast<long>(nframes) * 3 * height * out_w), 256, 0, st>>>(p);
  lr_height_kernel<<<blocks(static_cast<long>(nframes) * 3 * out_h * out_w), 256, 0, st>>>(p);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}
