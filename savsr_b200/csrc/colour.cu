// YUV 4:2:0 <-> packed 8-bit BGR on the device, so decoded video (NVDEC NV12 surfaces, ffmpeg yuv420p pipes) enters the uint8 BGR
// forward and its HR frames leave for an encoder without a colour conversion on the CPU.  Byte-exact with OpenCV 4's cv::cvtColor:
//   COLOR_YUV2BGR_I420 / COLOR_YUV2BGR_NV12: each pixel takes the chroma sample of its 2x2 block (nearest neighbour);
//   COLOR_BGR2YUV_I420: U and V come from the top-left pixel of each 2x2 block alone (no averaging).
// BT.601 limited range in 20-bit fixed point, constants in common.cuh.
//
// Plane description (both directions): the Y plane at `y` with row pitch y_pitch; chroma row r at u + r * c_pitch and v + r * c_pitch,
// sample c of that row at offset c * c_step (yuv420p: separate U and V planes, c_step 1; nv12: one interleaved plane, v = u + 1,
// c_step 2).  Frame k's planes are frame 0's plus k * frame_stride.  The BGR side is contiguous [n][h][w][3].
//
// Both kernels move bytes and do a few integer multiplies per pixel: bound by HBM.  Each thread owns four 2x2 chroma blocks (8 pixels of
// two rows), so every chroma sample is read or written once, and moves each row's bytes with the widest loads and stores the row's
// alignment allows (all rows of one frame row share it; see load_bytes / store_bytes).  A row's last group may be narrower (w % 8): it
// takes the byte-wise path.
#include "common.cuh"

namespace savsr {

constexpr int kYuvGroup = 8;   // pixels per thread and row: four 2x2 chroma blocks

// N bytes at p (N a multiple of 4) as N / 4 little-endian words, with 8-, 4-, 2- or 1-byte accesses as p's alignment allows.
template <int N>
__device__ __forceinline__ void load_bytes(const uint8_t* __restrict__ p, uint32_t (&w)[N / 4]) {
  const unsigned a = static_cast<unsigned>(reinterpret_cast<uintptr_t>(p));
  if (N % 8 == 0 && (a & 7) == 0) {
#pragma unroll
    for (int i = 0; i < N / 8; ++i) {
      const uint2 v = reinterpret_cast<const uint2*>(p)[i];
      w[2 * i] = v.x;
      w[2 * i + 1] = v.y;
    }
  } else if ((a & 3) == 0) {
#pragma unroll
    for (int i = 0; i < N / 4; ++i) w[i] = reinterpret_cast<const uint32_t*>(p)[i];
  } else if ((a & 1) == 0) {
    const uint16_t* q = reinterpret_cast<const uint16_t*>(p);
#pragma unroll
    for (int i = 0; i < N / 4; ++i) w[i] = q[2 * i] | (static_cast<uint32_t>(q[2 * i + 1]) << 16);
  } else {
#pragma unroll
    for (int i = 0; i < N / 4; ++i)
      w[i] = p[4 * i] | (p[4 * i + 1] << 8) | (p[4 * i + 2] << 16) | (static_cast<uint32_t>(p[4 * i + 3]) << 24);
  }
}

template <int N>
__device__ __forceinline__ void store_bytes(uint8_t* __restrict__ p, const uint32_t (&w)[N / 4]) {
  const unsigned a = static_cast<unsigned>(reinterpret_cast<uintptr_t>(p));
  if (N % 8 == 0 && (a & 7) == 0) {
#pragma unroll
    for (int i = 0; i < N / 8; ++i) reinterpret_cast<uint2*>(p)[i] = make_uint2(w[2 * i], w[2 * i + 1]);
  } else if ((a & 3) == 0) {
#pragma unroll
    for (int i = 0; i < N / 4; ++i) reinterpret_cast<uint32_t*>(p)[i] = w[i];
  } else if ((a & 1) == 0) {
    uint16_t* q = reinterpret_cast<uint16_t*>(p);
#pragma unroll
    for (int i = 0; i < N / 4; ++i) {
      q[2 * i] = static_cast<uint16_t>(w[i]);
      q[2 * i + 1] = static_cast<uint16_t>(w[i] >> 16);
    }
  } else {
#pragma unroll
    for (int i = 0; i < N; ++i) p[i] = static_cast<uint8_t>(w[i >> 2] >> (8 * (i & 3)));
  }
}

template <int N>
__device__ __forceinline__ int byte_at(const uint32_t (&w)[N], int i) { return (w[i >> 2] >> (8 * (i & 3))) & 0xff; }
template <int N>
__device__ __forceinline__ void put_byte(uint32_t (&w)[N], int i, int v) { w[i >> 2] |= static_cast<uint32_t>(v) << (8 * (i & 3)); }

__device__ __forceinline__ int sat_u8(int v) { return min(max(v, 0), 255); }

// The chroma terms of one 2x2 block (decode), shared by its four pixels.
struct Chroma {
  int r, g, b;
  Chroma() = default;
  __device__ __forceinline__ Chroma(int U, int V) {
    const int u = U - 128, v = V - 128;
    r = kYuvHalf + kYuvVR * v;
    g = kYuvHalf + kYuvVG * v + kYuvUG * u;
    b = kYuvHalf + kYuvUB * u;
  }
  __device__ __forceinline__ void bgr(int Y, int& B, int& G, int& R) const {
    const int y = max(Y - 16, 0) * kYuvY;
    B = sat_u8((y + b) >> kYuvShift);
    G = sat_u8((y + g) >> kYuvShift);
    R = sat_u8((y + r) >> kYuvShift);
  }
};
// Encode.  The results lie in [16, 235] (Y) and [16, 240] (U, V) for every 8-bit input, so no saturation is needed.
__device__ __forceinline__ int rgb_y(int R, int G, int B) { return (kRgbYR * R + kRgbYG * G + kRgbYB * B + (16 << kYuvShift) + kYuvHalf) >> kYuvShift; }
__device__ __forceinline__ int rgb_u(int R, int G, int B) { return (kRgbUR * R + kRgbUG * G + kRgbUB * B + (128 << kYuvShift) + kYuvHalf) >> kYuvShift; }
__device__ __forceinline__ int rgb_v(int R, int G, int B) { return (kRgbVR * R + kRgbVG * G + kRgbVB * B + (128 << kYuvShift) + kYuvHalf) >> kYuvShift; }

struct Yuv420Planes {
  uint8_t* y;
  uint8_t* u;
  uint8_t* v;
  int y_pitch, c_pitch, c_step;
  long long frame_stride;
};

// Work item idx -> frame f, row pair rp (rows 2 rp, 2 rp + 1), first pixel x0 of the group.
__device__ __forceinline__ void yuv_item(long long idx, int groups, int half_h, int& f, int& rp, int& x0) {
  const long long rest = idx / groups;
  x0 = static_cast<int>(idx - rest * groups) * kYuvGroup;
  rp = static_cast<int>(rest % half_h);
  f = static_cast<int>(rest / half_h);
}

__global__ void __launch_bounds__(256) yuv420_to_bgr_kernel(const Yuv420Planes p, int n, int h, int w, uint8_t* __restrict__ bgr) {
  const int groups = (w + kYuvGroup - 1) / kYuvGroup, half_h = h >> 1;
  const long long total = static_cast<long long>(n) * half_h * groups;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    int f, rp, x0;
    yuv_item(idx, groups, half_h, f, rp, x0);
    const long long fo = f * p.frame_stride;
    const uint8_t* y0 = p.y + fo + static_cast<long long>(2 * rp) * p.y_pitch + x0;
    const uint8_t* y1 = y0 + p.y_pitch;
    const long long co = fo + static_cast<long long>(rp) * p.c_pitch + (x0 >> 1) * p.c_step;
    const uint8_t* u = p.u + co;
    const uint8_t* v = p.v + co;
    uint8_t* o0 = bgr + ((static_cast<long long>(f) * h + 2 * rp) * w + x0) * 3;
    uint8_t* o1 = o0 + static_cast<long long>(w) * 3;
    if (x0 + kYuvGroup <= w) {
      uint32_t ya[2], yb[2], uw[1], vw[1];
      load_bytes<8>(y0, ya);
      load_bytes<8>(y1, yb);
      if (p.c_step == 1) {
        load_bytes<4>(u, uw);
        load_bytes<4>(v, vw);
      } else {                                     // nv12: U0 V0 U1 V1 U2 V2 U3 V3
        uint32_t uv[2];
        load_bytes<8>(u, uv);
        uw[0] = __byte_perm(uv[0], uv[1], 0x6420);
        vw[0] = __byte_perm(uv[0], uv[1], 0x7531);
      }
      Chroma c[kYuvGroup / 2];
#pragma unroll
      for (int k = 0; k < kYuvGroup / 2; ++k) c[k] = Chroma(byte_at(uw, k), byte_at(vw, k));
#pragma unroll
      for (int r = 0; r < 2; ++r) {                // one row at a time: the 24 output bytes of a row stay in 6 registers
        uint32_t o[6] = {0, 0, 0, 0, 0, 0};
#pragma unroll
        for (int j = 0; j < kYuvGroup; ++j) {
          int B, G, R;
          c[j >> 1].bgr(byte_at(r ? yb : ya, j), B, G, R);
          put_byte(o, 3 * j, B); put_byte(o, 3 * j + 1, G); put_byte(o, 3 * j + 2, R);
        }
        store_bytes<24>(r ? o1 : o0, o);
      }
    } else {
      for (int j = 0; x0 + j < w; j += 2) {
        const Chroma c(u[(j >> 1) * p.c_step], v[(j >> 1) * p.c_step]);
#pragma unroll
        for (int d = 0; d < 2; ++d) {
          int B, G, R;
          c.bgr(y0[j + d], B, G, R);
          o0[3 * (j + d)] = B; o0[3 * (j + d) + 1] = G; o0[3 * (j + d) + 2] = R;
          c.bgr(y1[j + d], B, G, R);
          o1[3 * (j + d)] = B; o1[3 * (j + d) + 1] = G; o1[3 * (j + d) + 2] = R;
        }
      }
    }
  }
}

__global__ void __launch_bounds__(256) bgr_to_yuv420_kernel(const uint8_t* __restrict__ bgr, int n, int h, int w, const Yuv420Planes p) {
  const int groups = (w + kYuvGroup - 1) / kYuvGroup, half_h = h >> 1;
  const long long total = static_cast<long long>(n) * half_h * groups;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    int f, rp, x0;
    yuv_item(idx, groups, half_h, f, rp, x0);
    const long long fo = f * p.frame_stride;
    uint8_t* y0 = p.y + fo + static_cast<long long>(2 * rp) * p.y_pitch + x0;
    uint8_t* y1 = y0 + p.y_pitch;
    const long long co = fo + static_cast<long long>(rp) * p.c_pitch + (x0 >> 1) * p.c_step;
    uint8_t* u = p.u + co;
    uint8_t* v = p.v + co;
    const uint8_t* i0 = bgr + ((static_cast<long long>(f) * h + 2 * rp) * w + x0) * 3;
    const uint8_t* i1 = i0 + static_cast<long long>(w) * 3;
    if (x0 + kYuvGroup <= w) {
      uint32_t ia[6], ib[6];
      load_bytes<24>(i0, ia);
      load_bytes<24>(i1, ib);
      uint32_t ya[2] = {0, 0}, yb[2] = {0, 0}, uw[1] = {0}, vw[1] = {0};
#pragma unroll
      for (int j = 0; j < kYuvGroup; ++j) {
        const int B = byte_at(ia, 3 * j), G = byte_at(ia, 3 * j + 1), R = byte_at(ia, 3 * j + 2);
        put_byte(ya, j, rgb_y(R, G, B));
        if ((j & 1) == 0) {                        // the top-left pixel of its 2x2 block
          put_byte(uw, j >> 1, rgb_u(R, G, B));
          put_byte(vw, j >> 1, rgb_v(R, G, B));
        }
        put_byte(yb, j, rgb_y(byte_at(ib, 3 * j + 2), byte_at(ib, 3 * j + 1), byte_at(ib, 3 * j)));
      }
      store_bytes<8>(y0, ya);
      store_bytes<8>(y1, yb);
      if (p.c_step == 1) {
        store_bytes<4>(u, uw);
        store_bytes<4>(v, vw);
      } else {
        const uint32_t uv[2] = {__byte_perm(uw[0], vw[0], 0x5140), __byte_perm(uw[0], vw[0], 0x7362)};
        store_bytes<8>(u, uv);
      }
    } else {
      for (int j = 0; x0 + j < w; j += 2) {
        const uint8_t* a = i0 + 3 * j;
        u[(j >> 1) * p.c_step] = static_cast<uint8_t>(rgb_u(a[2], a[1], a[0]));
        v[(j >> 1) * p.c_step] = static_cast<uint8_t>(rgb_v(a[2], a[1], a[0]));
#pragma unroll
        for (int d = 0; d < 2; ++d) {
          const uint8_t* q0 = i0 + 3 * (j + d);
          const uint8_t* q1 = i1 + 3 * (j + d);
          y0[j + d] = static_cast<uint8_t>(rgb_y(q0[2], q0[1], q0[0]));
          y1[j + d] = static_cast<uint8_t>(rgb_y(q1[2], q1[1], q1[0]));
        }
      }
    }
  }
}

// The checks both entry points make before any launch.
static int check_yuv420(const char* fn, int n, int h, int w, int y_pitch, int c_pitch, int c_step, long long frame_stride) {
  SAVSR_REQUIRE(n >= 0 && h > 0 && w > 0, "%s: bad shape n=%d h=%d w=%d", fn, n, h, w);
  SAVSR_REQUIRE(h % 2 == 0 && w % 2 == 0, "%s: YUV 4:2:0 needs an even frame size, got %dx%d", fn, h, w);
  SAVSR_REQUIRE(c_step == 1 || c_step == 2, "%s: c_step must be 1 (yuv420p) or 2 (nv12), got %d", fn, c_step);
  SAVSR_REQUIRE(y_pitch >= w, "%s: y_pitch %d < width %d", fn, y_pitch, w);
  SAVSR_REQUIRE(c_pitch >= c_step * (w / 2), "%s: c_pitch %d < chroma row of %d bytes", fn, c_pitch, c_step * (w / 2));
  SAVSR_REQUIRE(frame_stride >= 0, "%s: negative frame_stride %lld", fn, frame_stride);
  return 0;
}

static unsigned yuv_blocks(const savsr_ctx* ctx, int n, int h, int w) {
  const long long items = static_cast<long long>(n) * (h / 2) * ((w + kYuvGroup - 1) / kYuvGroup);
  const long long b = (items + 255) / 256, cap = 16LL * ctx->sm_count;
  return static_cast<unsigned>(b < cap ? b : cap);
}

}  // namespace savsr

using namespace savsr;

extern "C" int savsr_yuv420_to_bgr(savsr_ctx* ctx, const uint8_t* y, int y_pitch, const uint8_t* u, const uint8_t* v, int c_pitch,
                                   int c_step, int64_t frame_stride, int n, int h, int w, uint8_t* bgr, savsr_stream st) {
  SAVSR_REQUIRE(ctx && y && u && v && bgr, "savsr_yuv420_to_bgr: null pointer");
  if (check_yuv420("savsr_yuv420_to_bgr", n, h, w, y_pitch, c_pitch, c_step, frame_stride)) return 1;
  if (n == 0) return 0;
  DeviceGuard guard(ctx->device);
  const Yuv420Planes p{const_cast<uint8_t*>(y), const_cast<uint8_t*>(u), const_cast<uint8_t*>(v), y_pitch, c_pitch, c_step, frame_stride};
  yuv420_to_bgr_kernel<<<yuv_blocks(ctx, n, h, w), 256, 0, static_cast<cudaStream_t>(st)>>>(p, n, h, w, bgr);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int savsr_bgr_to_yuv420(savsr_ctx* ctx, const uint8_t* bgr, int n, int h, int w, uint8_t* y, int y_pitch, uint8_t* u, uint8_t* v,
                                   int c_pitch, int c_step, int64_t frame_stride, savsr_stream st) {
  SAVSR_REQUIRE(ctx && bgr && y && u && v, "savsr_bgr_to_yuv420: null pointer");
  if (check_yuv420("savsr_bgr_to_yuv420", n, h, w, y_pitch, c_pitch, c_step, frame_stride)) return 1;
  if (n == 0) return 0;
  DeviceGuard guard(ctx->device);
  const Yuv420Planes p{y, u, v, y_pitch, c_pitch, c_step, frame_stride};
  bgr_to_yuv420_kernel<<<yuv_blocks(ctx, n, h, w), 256, 0, static_cast<cudaStream_t>(st)>>>(bgr, n, h, w, p);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}
