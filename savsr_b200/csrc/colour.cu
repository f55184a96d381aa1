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
//
// 10-bit YUV 4:2:0 <-> 16-bit BGR (yuv420p10le, p010 <-> bgr48): the same matrix, chroma handling and work split in fixed-point forms
// rescaled to the deeper samples (common.cuh), with pitches and frame strides in uint16 elements.  A thread's rows are 16 bytes of Y and
// 48 of BGR, so 16-byte accesses are used where the row's alignment allows.  widen_u8_to_u16 brings 8-bit BGR frames into a 16-bit ring.
//
// Other colour matrices and ranges (the _cs entry points): the same four kernel bodies over the H.273 map of one (colorspace, range)
// pair, one instantiation per pair with the coefficients of common.cuh's kYuvCoeffs8 / kYuvCoeffs10 as compile-time constants.
#include "common.cuh"

namespace savsr {

constexpr int kYuvGroup = 8;   // pixels per thread and row: four 2x2 chroma blocks

// N bytes at p (N a multiple of 4) as N / 4 little-endian words, with 8-, 4-, 2- or 1-byte accesses as p's alignment allows.
template <int N>
__device__ __forceinline__ void load_bytes(const uint8_t* __restrict__ p, uint32_t (&w)[N / 4]) {
  const unsigned a = static_cast<unsigned>(reinterpret_cast<uintptr_t>(p));
  if (N % 16 == 0 && (a & 15) == 0) {
#pragma unroll
    for (int i = 0; i < N / 16; ++i) {
      const uint4 v = reinterpret_cast<const uint4*>(p)[i];
      w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w;
    }
  } else if (N % 8 == 0 && (a & 7) == 0) {
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
  if (N % 16 == 0 && (a & 15) == 0) {
#pragma unroll
    for (int i = 0; i < N / 16; ++i) reinterpret_cast<uint4*>(p)[i] = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
  } else if (N % 8 == 0 && (a & 7) == 0) {
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

// The kernel bodies are written over a pixel map: chroma(U, V) once per 2x2 block and pixel(c, Y, B, G, R) per pixel (decode), and
// y, u, v of (R, G, B) (encode).  Cv2Map8: the cv2-exact BT.601 limited-range functions above.  CsMap8<CS, RNG>: the H.273 map of
// one (matrix, range) pair, its coefficients compile-time constants from kYuvCoeffs8 (one instantiation per pair: with the
// coefficients passed by value instead, the 8-bit encode needed 62 registers instead of 40 and ran 17 % slower at 1080p x 26).
struct Cv2Map8 {
  using Chroma = savsr::Chroma;
  __device__ __forceinline__ Chroma chroma(int U, int V) const { return Chroma(U, V); }
  __device__ __forceinline__ void pixel(const Chroma& c, int Y, int& B, int& G, int& R) const { c.bgr(Y, B, G, R); }
  __device__ __forceinline__ int y(int R, int G, int B) const { return rgb_y(R, G, B); }
  __device__ __forceinline__ int u(int R, int G, int B) const { return rgb_u(R, G, B); }
  __device__ __forceinline__ int v(int R, int G, int B) const { return rgb_v(R, G, B); }
};

template <int CS, int RNG>
struct CsMap8 {
  struct Chroma { int r, g, b; };
  static constexpr YuvCoeffs k = kYuvCoeffs8[CS][RNG];
  static constexpr int kHalf = 1 << (kCs8Shift - 1);
  __device__ __forceinline__ Chroma chroma(int U, int V) const {
    const int u = U - 128, v = V - 128;
    return {kHalf + k.dvr * v, kHalf + k.dvg * v + k.dug * u, kHalf + k.dub * u};
  }
  __device__ __forceinline__ void pixel(const Chroma& c, int Y, int& B, int& G, int& R) const {
    const int y = (Y - k.y0) * k.dy;
    B = sat_u8((y + c.b) >> kCs8Shift);
    G = sat_u8((y + c.g) >> kCs8Shift);
    R = sat_u8((y + c.r) >> kCs8Shift);
  }
  __device__ __forceinline__ int y(int R, int G, int B) const { return sat_u8(k.y0 + ((k.eyr * R + k.eyg * G + k.eyb * B + kHalf) >> kCs8Shift)); }
  __device__ __forceinline__ int u(int R, int G, int B) const { return sat_u8(128 + ((k.eur * R + k.eug * G + k.eub * B + kHalf) >> kCs8Shift)); }
  __device__ __forceinline__ int v(int R, int G, int B) const { return sat_u8(128 + ((k.evr * R + k.evg * G + k.evb * B + kHalf) >> kCs8Shift)); }
};

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

template <class Map>
__device__ __forceinline__ void yuv420_to_bgr_body(const Yuv420Planes& p, int n, int h, int w, uint8_t* __restrict__ bgr, const Map& m) {
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
      typename Map::Chroma c[kYuvGroup / 2];
#pragma unroll
      for (int k = 0; k < kYuvGroup / 2; ++k) c[k] = m.chroma(byte_at(uw, k), byte_at(vw, k));
#pragma unroll
      for (int r = 0; r < 2; ++r) {                // one row at a time: the 24 output bytes of a row stay in 6 registers
        uint32_t o[6] = {0, 0, 0, 0, 0, 0};
#pragma unroll
        for (int j = 0; j < kYuvGroup; ++j) {
          int B, G, R;
          m.pixel(c[j >> 1], byte_at(r ? yb : ya, j), B, G, R);
          put_byte(o, 3 * j, B); put_byte(o, 3 * j + 1, G); put_byte(o, 3 * j + 2, R);
        }
        store_bytes<24>(r ? o1 : o0, o);
      }
    } else {
      for (int j = 0; x0 + j < w; j += 2) {
        const typename Map::Chroma c = m.chroma(u[(j >> 1) * p.c_step], v[(j >> 1) * p.c_step]);
#pragma unroll
        for (int d = 0; d < 2; ++d) {
          int B, G, R;
          m.pixel(c, y0[j + d], B, G, R);
          o0[3 * (j + d)] = B; o0[3 * (j + d) + 1] = G; o0[3 * (j + d) + 2] = R;
          m.pixel(c, y1[j + d], B, G, R);
          o1[3 * (j + d)] = B; o1[3 * (j + d) + 1] = G; o1[3 * (j + d) + 2] = R;
        }
      }
    }
  }
}

__global__ void __launch_bounds__(256) yuv420_to_bgr_kernel(const Yuv420Planes p, int n, int h, int w, uint8_t* __restrict__ bgr) {
  yuv420_to_bgr_body(p, n, h, w, bgr, Cv2Map8{});
}
template <int CS, int RNG>
__global__ void __launch_bounds__(256) yuv420_to_bgr_cs_kernel(const Yuv420Planes p, int n, int h, int w, uint8_t* __restrict__ bgr) {
  yuv420_to_bgr_body(p, n, h, w, bgr, CsMap8<CS, RNG>{});
}

template <class Map>
__device__ __forceinline__ void bgr_to_yuv420_body(const uint8_t* __restrict__ bgr, int n, int h, int w, const Yuv420Planes& p, const Map& m) {
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
        put_byte(ya, j, m.y(R, G, B));
        if ((j & 1) == 0) {                        // the top-left pixel of its 2x2 block
          put_byte(uw, j >> 1, m.u(R, G, B));
          put_byte(vw, j >> 1, m.v(R, G, B));
        }
        put_byte(yb, j, m.y(byte_at(ib, 3 * j + 2), byte_at(ib, 3 * j + 1), byte_at(ib, 3 * j)));
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
        u[(j >> 1) * p.c_step] = static_cast<uint8_t>(m.u(a[2], a[1], a[0]));
        v[(j >> 1) * p.c_step] = static_cast<uint8_t>(m.v(a[2], a[1], a[0]));
#pragma unroll
        for (int d = 0; d < 2; ++d) {
          const uint8_t* q0 = i0 + 3 * (j + d);
          const uint8_t* q1 = i1 + 3 * (j + d);
          y0[j + d] = static_cast<uint8_t>(m.y(q0[2], q0[1], q0[0]));
          y1[j + d] = static_cast<uint8_t>(m.y(q1[2], q1[1], q1[0]));
        }
      }
    }
  }
}

__global__ void __launch_bounds__(256) bgr_to_yuv420_kernel(const uint8_t* __restrict__ bgr, int n, int h, int w, const Yuv420Planes p) {
  bgr_to_yuv420_body(bgr, n, h, w, p, Cv2Map8{});
}
template <int CS, int RNG>
__global__ void __launch_bounds__(256) bgr_to_yuv420_cs_kernel(const uint8_t* __restrict__ bgr, int n, int h, int w, const Yuv420Planes p) {
  bgr_to_yuv420_body(bgr, n, h, w, p, CsMap8<CS, RNG>{});
}

// ------------------------------------------------------------------------------------------------ 10-bit YUV <-> 16-bit BGR
template <int N>
__device__ __forceinline__ int half_at(const uint32_t (&w)[N], int i) { return (w[i >> 1] >> (16 * (i & 1))) & 0xffff; }
template <int N>
__device__ __forceinline__ void put_half(uint32_t (&w)[N], int i, int v) { w[i >> 1] |= static_cast<uint32_t>(v) << (16 * (i & 1)); }

__device__ __forceinline__ int sat_u16(int v) { return min(max(v, 0), 65535); }
// A 10-bit sample from its 16-bit container: p010 keeps it in bits 6-15, yuv420p10le in bits 0-9.
__device__ __forceinline__ int sample10(int s, int msb) { return msb ? s >> 6 : s & 0x3ff; }

struct Chroma10 {
  long long r, g, b;
  Chroma10() = default;
  __device__ __forceinline__ Chroma10(int U, int V) {
    const int u = U - 512, v = V - 512;
    r = kYuv10Half + static_cast<long long>(kYuv10VR) * v;
    g = kYuv10Half + static_cast<long long>(kYuv10VG) * v + static_cast<long long>(kYuv10UG) * u;
    b = kYuv10Half + static_cast<long long>(kYuv10UB) * u;
  }
  __device__ __forceinline__ void bgr(int Y, int& B, int& G, int& R) const {
    const long long y = static_cast<long long>(max(Y - 64, 0)) * kYuv10Y;
    B = sat_u16(static_cast<int>((y + b) >> kYuv10Shift));
    G = sat_u16(static_cast<int>((y + g) >> kYuv10Shift));
    R = sat_u16(static_cast<int>((y + r) >> kYuv10Shift));
  }
};
__device__ __forceinline__ int rgb_y10(int R, int G, int B) {
  return (kRgb10YR * R + kRgb10YG * G + kRgb10YB * B + (64 << kRgb10Shift) + kRgb10Half) >> kRgb10Shift;
}
__device__ __forceinline__ int rgb_u10(int R, int G, int B) {
  return (kRgb10UR * R + kRgb10UG * G + kRgb10UB * B + (512 << kRgb10Shift) + kRgb10Half) >> kRgb10Shift;
}
__device__ __forceinline__ int rgb_v10(int R, int G, int B) {
  return (kRgb10VR * R + kRgb10VG * G + kRgb10VB * B + (512 << kRgb10Shift) + kRgb10Half) >> kRgb10Shift;
}
__device__ __forceinline__ int sat_u10(int v) { return min(max(v, 0), 1023); }

// The 10-bit pixel maps, as Cv2Map8 / CsMap8 (10-bit YUV samples, 16-bit BGR; coefficients from kYuvCoeffs10).
struct Cv2Map10 {
  using Chroma = Chroma10;
  __device__ __forceinline__ Chroma chroma(int U, int V) const { return Chroma(U, V); }
  __device__ __forceinline__ void pixel(const Chroma& c, int Y, int& B, int& G, int& R) const { c.bgr(Y, B, G, R); }
  __device__ __forceinline__ int y(int R, int G, int B) const { return rgb_y10(R, G, B); }
  __device__ __forceinline__ int u(int R, int G, int B) const { return rgb_u10(R, G, B); }
  __device__ __forceinline__ int v(int R, int G, int B) const { return rgb_v10(R, G, B); }
};

template <int CS, int RNG>
struct CsMap10 {
  struct Chroma { long long r, g, b; };
  static constexpr YuvCoeffs k = kYuvCoeffs10[CS][RNG];
  static constexpr long long kDecHalf = 1LL << (kCs10DecShift - 1);
  static constexpr int kEncHalf = 1 << (kCs10EncShift - 1);
  __device__ __forceinline__ Chroma chroma(int U, int V) const {
    const int u = U - 512, v = V - 512;
    return {kDecHalf + static_cast<long long>(k.dvr) * v, kDecHalf + static_cast<long long>(k.dvg) * v + static_cast<long long>(k.dug) * u,
            kDecHalf + static_cast<long long>(k.dub) * u};
  }
  __device__ __forceinline__ void pixel(const Chroma& c, int Y, int& B, int& G, int& R) const {
    const long long y = static_cast<long long>(Y - k.y0) * k.dy;
    B = sat_u16(static_cast<int>((y + c.b) >> kCs10DecShift));
    G = sat_u16(static_cast<int>((y + c.g) >> kCs10DecShift));
    R = sat_u16(static_cast<int>((y + c.r) >> kCs10DecShift));
  }
  __device__ __forceinline__ int y(int R, int G, int B) const {
    return sat_u10(k.y0 + ((k.eyr * R + k.eyg * G + k.eyb * B + kEncHalf) >> kCs10EncShift));
  }
  __device__ __forceinline__ int u(int R, int G, int B) const {
    return sat_u10(512 + ((k.eur * R + k.eug * G + k.eub * B + kEncHalf) >> kCs10EncShift));
  }
  __device__ __forceinline__ int v(int R, int G, int B) const {
    return sat_u10(512 + ((k.evr * R + k.evg * G + k.evb * B + kEncHalf) >> kCs10EncShift));
  }
};

// Yuv420Planes in uint16 elements, plus where the 10 bits sit (msb: 1 for p010, 0 for yuv420p10le).
struct Yuv420Planes16 {
  uint16_t* y;
  uint16_t* u;
  uint16_t* v;
  int y_pitch, c_pitch, c_step;
  long long frame_stride;
  int msb;
};

template <class T>
__device__ __forceinline__ const uint8_t* as_bytes(const T* p) { return reinterpret_cast<const uint8_t*>(p); }
template <class T>
__device__ __forceinline__ uint8_t* as_bytes(T* p) { return reinterpret_cast<uint8_t*>(p); }

template <class Map>
__device__ __forceinline__ void yuv420_10_to_bgr48_body(const Yuv420Planes16& p, int n, int h, int w, uint16_t* __restrict__ bgr, const Map& m) {
  const int groups = (w + kYuvGroup - 1) / kYuvGroup, half_h = h >> 1;
  const long long total = static_cast<long long>(n) * half_h * groups;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    int f, rp, x0;
    yuv_item(idx, groups, half_h, f, rp, x0);
    const long long fo = f * p.frame_stride;
    const uint16_t* y0 = p.y + fo + static_cast<long long>(2 * rp) * p.y_pitch + x0;
    const uint16_t* y1 = y0 + p.y_pitch;
    const long long co = fo + static_cast<long long>(rp) * p.c_pitch + (x0 >> 1) * p.c_step;
    const uint16_t* u = p.u + co;
    const uint16_t* v = p.v + co;
    uint16_t* o0 = bgr + ((static_cast<long long>(f) * h + 2 * rp) * w + x0) * 3;
    uint16_t* o1 = o0 + static_cast<long long>(w) * 3;
    if (x0 + kYuvGroup <= w) {
      uint32_t ya[4], yb[4], uw[2], vw[2];
      load_bytes<16>(as_bytes(y0), ya);
      load_bytes<16>(as_bytes(y1), yb);
      if (p.c_step == 1) {
        load_bytes<8>(as_bytes(u), uw);
        load_bytes<8>(as_bytes(v), vw);
      } else {                                     // p010: U0 V0 U1 V1 U2 V2 U3 V3, 16 bits each
        uint32_t uv[4];
        load_bytes<16>(as_bytes(u), uv);
        uw[0] = __byte_perm(uv[0], uv[1], 0x5410); uw[1] = __byte_perm(uv[2], uv[3], 0x5410);
        vw[0] = __byte_perm(uv[0], uv[1], 0x7632); vw[1] = __byte_perm(uv[2], uv[3], 0x7632);
      }
      typename Map::Chroma c[kYuvGroup / 2];
#pragma unroll
      for (int k = 0; k < kYuvGroup / 2; ++k) c[k] = m.chroma(sample10(half_at(uw, k), p.msb), sample10(half_at(vw, k), p.msb));
#pragma unroll
      for (int r = 0; r < 2; ++r) {                // one row at a time: the 48 output bytes of a row stay in 12 registers
        uint32_t o[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
        for (int j = 0; j < kYuvGroup; ++j) {
          int B, G, R;
          m.pixel(c[j >> 1], sample10(half_at(r ? yb : ya, j), p.msb), B, G, R);
          put_half(o, 3 * j, B); put_half(o, 3 * j + 1, G); put_half(o, 3 * j + 2, R);
        }
        store_bytes<48>(as_bytes(r ? o1 : o0), o);
      }
    } else {
      for (int j = 0; x0 + j < w; j += 2) {
        const typename Map::Chroma c = m.chroma(sample10(u[(j >> 1) * p.c_step], p.msb), sample10(v[(j >> 1) * p.c_step], p.msb));
#pragma unroll
        for (int d = 0; d < 2; ++d) {
          int B, G, R;
          m.pixel(c, sample10(y0[j + d], p.msb), B, G, R);
          o0[3 * (j + d)] = B; o0[3 * (j + d) + 1] = G; o0[3 * (j + d) + 2] = R;
          m.pixel(c, sample10(y1[j + d], p.msb), B, G, R);
          o1[3 * (j + d)] = B; o1[3 * (j + d) + 1] = G; o1[3 * (j + d) + 2] = R;
        }
      }
    }
  }
}

__global__ void __launch_bounds__(256) yuv420_10_to_bgr48_kernel(const Yuv420Planes16 p, int n, int h, int w, uint16_t* __restrict__ bgr) {
  yuv420_10_to_bgr48_body(p, n, h, w, bgr, Cv2Map10{});
}
template <int CS, int RNG>
__global__ void __launch_bounds__(256) yuv420_10_to_bgr48_cs_kernel(const Yuv420Planes16 p, int n, int h, int w, uint16_t* __restrict__ bgr) {
  yuv420_10_to_bgr48_body(p, n, h, w, bgr, CsMap10<CS, RNG>{});
}

template <class Map>
__device__ __forceinline__ void bgr48_to_yuv420_10_body(const uint16_t* __restrict__ bgr, int n, int h, int w, const Yuv420Planes16& p,
                                                        const Map& m) {
  const int groups = (w + kYuvGroup - 1) / kYuvGroup, half_h = h >> 1;
  const long long total = static_cast<long long>(n) * half_h * groups;
  const int sh = p.msb ? 6 : 0;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    int f, rp, x0;
    yuv_item(idx, groups, half_h, f, rp, x0);
    const long long fo = f * p.frame_stride;
    uint16_t* y0 = p.y + fo + static_cast<long long>(2 * rp) * p.y_pitch + x0;
    uint16_t* y1 = y0 + p.y_pitch;
    const long long co = fo + static_cast<long long>(rp) * p.c_pitch + (x0 >> 1) * p.c_step;
    uint16_t* u = p.u + co;
    uint16_t* v = p.v + co;
    const uint16_t* i0 = bgr + ((static_cast<long long>(f) * h + 2 * rp) * w + x0) * 3;
    const uint16_t* i1 = i0 + static_cast<long long>(w) * 3;
    if (x0 + kYuvGroup <= w) {
      uint32_t ia[12], ib[12];
      load_bytes<48>(as_bytes(i0), ia);
      load_bytes<48>(as_bytes(i1), ib);
      uint32_t ya[4] = {0, 0, 0, 0}, yb[4] = {0, 0, 0, 0}, uw[2] = {0, 0}, vw[2] = {0, 0};
#pragma unroll
      for (int j = 0; j < kYuvGroup; ++j) {
        const int B = half_at(ia, 3 * j), G = half_at(ia, 3 * j + 1), R = half_at(ia, 3 * j + 2);
        put_half(ya, j, m.y(R, G, B) << sh);
        if ((j & 1) == 0) {                        // the top-left pixel of its 2x2 block
          put_half(uw, j >> 1, m.u(R, G, B) << sh);
          put_half(vw, j >> 1, m.v(R, G, B) << sh);
        }
        put_half(yb, j, m.y(half_at(ib, 3 * j + 2), half_at(ib, 3 * j + 1), half_at(ib, 3 * j)) << sh);
      }
      store_bytes<16>(as_bytes(y0), ya);
      store_bytes<16>(as_bytes(y1), yb);
      if (p.c_step == 1) {
        store_bytes<8>(as_bytes(u), uw);
        store_bytes<8>(as_bytes(v), vw);
      } else {
        const uint32_t uv[4] = {__byte_perm(uw[0], vw[0], 0x5410), __byte_perm(uw[0], vw[0], 0x7632),
                                __byte_perm(uw[1], vw[1], 0x5410), __byte_perm(uw[1], vw[1], 0x7632)};
        store_bytes<16>(as_bytes(u), uv);
      }
    } else {
      for (int j = 0; x0 + j < w; j += 2) {
        const uint16_t* a = i0 + 3 * j;
        u[(j >> 1) * p.c_step] = static_cast<uint16_t>(m.u(a[2], a[1], a[0]) << sh);
        v[(j >> 1) * p.c_step] = static_cast<uint16_t>(m.v(a[2], a[1], a[0]) << sh);
#pragma unroll
        for (int d = 0; d < 2; ++d) {
          const uint16_t* q0 = i0 + 3 * (j + d);
          const uint16_t* q1 = i1 + 3 * (j + d);
          y0[j + d] = static_cast<uint16_t>(m.y(q0[2], q0[1], q0[0]) << sh);
          y1[j + d] = static_cast<uint16_t>(m.y(q1[2], q1[1], q1[0]) << sh);
        }
      }
    }
  }
}

__global__ void __launch_bounds__(256) bgr48_to_yuv420_10_kernel(const uint16_t* __restrict__ bgr, int n, int h, int w, const Yuv420Planes16 p) {
  bgr48_to_yuv420_10_body(bgr, n, h, w, p, Cv2Map10{});
}
template <int CS, int RNG>
__global__ void __launch_bounds__(256) bgr48_to_yuv420_10_cs_kernel(const uint16_t* __restrict__ bgr, int n, int h, int w, const Yuv420Planes16 p) {
  bgr48_to_yuv420_10_body(bgr, n, h, w, p, CsMap10<CS, RNG>{});
}

// x 257 (u -> u << 8 | u): 16 bytes in, 32 out per thread where both pointers are 16-byte aligned, one byte at a time otherwise.
__global__ void __launch_bounds__(256) widen_u8_to_u16_kernel(const uint8_t* __restrict__ src, uint16_t* __restrict__ dst, long long count) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  const long long first = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  const bool vec = ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0;
  const long long groups = vec ? count / 16 : 0;
  for (long long i = first; i < groups; i += stride) {
    const uint4 s = reinterpret_cast<const uint4*>(src)[i];
    uint4* d = reinterpret_cast<uint4*>(dst) + 2 * i;
    d[0] = make_uint4(__byte_perm(s.x, 0, 0x1100), __byte_perm(s.x, 0, 0x3322), __byte_perm(s.y, 0, 0x1100), __byte_perm(s.y, 0, 0x3322));
    d[1] = make_uint4(__byte_perm(s.z, 0, 0x1100), __byte_perm(s.z, 0, 0x3322), __byte_perm(s.w, 0, 0x1100), __byte_perm(s.w, 0, 0x3322));
  }
  for (long long i = groups * 16 + first; i < count; i += stride) dst[i] = static_cast<uint16_t>(src[i] * 257);
}

// ------------------------------------------------------------------------------------------------ YUV 4:2:2 <-> BGR
// 4:2:2 halves the chroma horizontally only: frame row r has chroma row r, and each horizontal pixel pair shares one (U, V).  Decoding
// gives both pixels of a pair its chroma (cv2's COLOR_YUV2BGR_YUYV / _UYVY); encoding takes U and V from the pair's left pixel, the
// co-sited position of H.264, HEVC and ProRes 4:2:2 and the 4:2:0 encode's point-sampling rule, so a 4:2:0 encode is the 4:2:2 encode
// with its odd chroma rows dropped.  (cv2's COLOR_BGR2YUV_YUYV averages the pair's chroma and rounds Y otherwise: it is not this.)
// The pixel maps are those of 4:2:0.  A thread owns kYuvGroup pixels of one row (four pairs), so odd heights need nothing special;
// every sample is read or written once, with the widest accesses the row's alignment allows, and a row's last w % 8 pixels take the
// sample-wise path.
//
// Plane description: Yuv420Planes plus y_step, the distance between Y samples of a row: 1 for the planar layout (yuv422p: c_step 1) and
// the semi-planar one (nv16: one interleaved U, V plane, v = u + 1, c_step 2), 2 for the packed ones, whose y, u and v point into the
// same rows of 4-byte macropixels (c_step 4): yuyv422 Y0 U0 Y1 V0 (u = y + 1, v = y + 3), uyvy422 U0 Y0 V0 Y1 (u = y - 1, v = y + 1).
struct Yuv422Planes {
  uint8_t* y;
  uint8_t* u;
  uint8_t* v;
  int y_pitch, y_step, c_pitch, c_step;
  long long frame_stride;
};

template <class Map>
__device__ __forceinline__ void yuv422_to_bgr_body(const Yuv422Planes& p, int n, int h, int w, uint8_t* __restrict__ bgr, const Map& m) {
  const int groups = (w + kYuvGroup - 1) / kYuvGroup;
  const long long total = static_cast<long long>(n) * h * groups;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    int f, r, x0;
    yuv_item(idx, groups, h, f, r, x0);
    const long long fo = f * p.frame_stride;
    const uint8_t* y = p.y + fo + static_cast<long long>(r) * p.y_pitch + x0 * p.y_step;
    const long long co = fo + static_cast<long long>(r) * p.c_pitch + (x0 >> 1) * p.c_step;
    const uint8_t* u = p.u + co;
    const uint8_t* v = p.v + co;
    uint8_t* o = bgr + ((static_cast<long long>(f) * h + r) * w + x0) * 3;
    if (x0 + kYuvGroup <= w) {
      uint32_t yw[2], uw[1], vw[1];
      if (p.y_step == 2) {                         // four macropixels, from whichever of y and u comes first
        const bool uyvy = u < y;
        uint32_t q[4];
        load_bytes<16>(uyvy ? u : y, q);
        const unsigned sy = uyvy ? 0x7531 : 0x6420, sc = uyvy ? 0x6420 : 0x7531;
        yw[0] = __byte_perm(q[0], q[1], sy);
        yw[1] = __byte_perm(q[2], q[3], sy);
        const uint32_t c01 = __byte_perm(q[0], q[1], sc), c23 = __byte_perm(q[2], q[3], sc);     // U0 V0 U1 V1, U2 V2 U3 V3
        uw[0] = __byte_perm(c01, c23, 0x6420);
        vw[0] = __byte_perm(c01, c23, 0x7531);
      } else {
        load_bytes<8>(y, yw);
        if (p.c_step == 1) {
          load_bytes<4>(u, uw);
          load_bytes<4>(v, vw);
        } else {                                   // nv16: U0 V0 U1 V1 U2 V2 U3 V3
          uint32_t uv[2];
          load_bytes<8>(u, uv);
          uw[0] = __byte_perm(uv[0], uv[1], 0x6420);
          vw[0] = __byte_perm(uv[0], uv[1], 0x7531);
        }
      }
      typename Map::Chroma c[kYuvGroup / 2];
#pragma unroll
      for (int k = 0; k < kYuvGroup / 2; ++k) c[k] = m.chroma(byte_at(uw, k), byte_at(vw, k));
      uint32_t out[6] = {0, 0, 0, 0, 0, 0};
#pragma unroll
      for (int j = 0; j < kYuvGroup; ++j) {
        int B, G, R;
        m.pixel(c[j >> 1], byte_at(yw, j), B, G, R);
        put_byte(out, 3 * j, B); put_byte(out, 3 * j + 1, G); put_byte(out, 3 * j + 2, R);
      }
      store_bytes<24>(o, out);
    } else {
      for (int j = 0; x0 + j < w; j += 2) {
        const typename Map::Chroma c = m.chroma(u[(j >> 1) * p.c_step], v[(j >> 1) * p.c_step]);
#pragma unroll
        for (int d = 0; d < 2; ++d) {
          int B, G, R;
          m.pixel(c, y[(j + d) * p.y_step], B, G, R);
          o[3 * (j + d)] = B; o[3 * (j + d) + 1] = G; o[3 * (j + d) + 2] = R;
        }
      }
    }
  }
}

template <class Map>
__global__ void __launch_bounds__(256) yuv422_to_bgr_kernel(const Yuv422Planes p, int n, int h, int w, uint8_t* __restrict__ bgr) {
  yuv422_to_bgr_body(p, n, h, w, bgr, Map{});
}

template <class Map>
__device__ __forceinline__ void bgr_to_yuv422_body(const uint8_t* __restrict__ bgr, int n, int h, int w, const Yuv422Planes& p, const Map& m) {
  const int groups = (w + kYuvGroup - 1) / kYuvGroup;
  const long long total = static_cast<long long>(n) * h * groups;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    int f, r, x0;
    yuv_item(idx, groups, h, f, r, x0);
    const long long fo = f * p.frame_stride;
    uint8_t* y = p.y + fo + static_cast<long long>(r) * p.y_pitch + x0 * p.y_step;
    const long long co = fo + static_cast<long long>(r) * p.c_pitch + (x0 >> 1) * p.c_step;
    uint8_t* u = p.u + co;
    uint8_t* v = p.v + co;
    const uint8_t* in = bgr + ((static_cast<long long>(f) * h + r) * w + x0) * 3;
    if (x0 + kYuvGroup <= w) {
      uint32_t ia[6];
      load_bytes<24>(in, ia);
      uint32_t yw[2] = {0, 0}, uw[1] = {0}, vw[1] = {0};
#pragma unroll
      for (int j = 0; j < kYuvGroup; ++j) {
        const int B = byte_at(ia, 3 * j), G = byte_at(ia, 3 * j + 1), R = byte_at(ia, 3 * j + 2);
        put_byte(yw, j, m.y(R, G, B));
        if ((j & 1) == 0) {                        // the left pixel of its pair
          put_byte(uw, j >> 1, m.u(R, G, B));
          put_byte(vw, j >> 1, m.v(R, G, B));
        }
      }
      if (p.y_step == 2) {
        const bool uyvy = u < y;
        const uint32_t c01 = __byte_perm(uw[0], vw[0], 0x5140), c23 = __byte_perm(uw[0], vw[0], 0x7362);   // U0 V0 U1 V1, U2 V2 U3 V3
        const unsigned s0 = uyvy ? 0x1504 : 0x5140, s1 = uyvy ? 0x3726 : 0x7362;
        const uint32_t q[4] = {__byte_perm(yw[0], c01, s0), __byte_perm(yw[0], c01, s1), __byte_perm(yw[1], c23, s0),
                               __byte_perm(yw[1], c23, s1)};
        store_bytes<16>(uyvy ? u : y, q);
      } else {
        store_bytes<8>(y, yw);
        if (p.c_step == 1) {
          store_bytes<4>(u, uw);
          store_bytes<4>(v, vw);
        } else {
          const uint32_t uv[2] = {__byte_perm(uw[0], vw[0], 0x5140), __byte_perm(uw[0], vw[0], 0x7362)};
          store_bytes<8>(u, uv);
        }
      }
    } else {
      for (int j = 0; x0 + j < w; j += 2) {
        const uint8_t* a = in + 3 * j;
        u[(j >> 1) * p.c_step] = static_cast<uint8_t>(m.u(a[2], a[1], a[0]));
        v[(j >> 1) * p.c_step] = static_cast<uint8_t>(m.v(a[2], a[1], a[0]));
#pragma unroll
        for (int d = 0; d < 2; ++d) {
          const uint8_t* q = in + 3 * (j + d);
          y[(j + d) * p.y_step] = static_cast<uint8_t>(m.y(q[2], q[1], q[0]));
        }
      }
    }
  }
}

template <class Map>
__global__ void __launch_bounds__(256) bgr_to_yuv422_kernel(const uint8_t* __restrict__ bgr, int n, int h, int w, const Yuv422Planes p) {
  bgr_to_yuv422_body(bgr, n, h, w, p, Map{});
}

// 10-bit 4:2:2 (yuv422p10le, p210): Yuv420Planes16 describes the planes, y_step is 1.  A thread's row is 16 bytes of Y, 8 of U and of V
// (or 16 of interleaved U, V) and 48 of BGR.
template <class Map>
__device__ __forceinline__ void yuv422_10_to_bgr48_body(const Yuv420Planes16& p, int n, int h, int w, uint16_t* __restrict__ bgr, const Map& m) {
  const int groups = (w + kYuvGroup - 1) / kYuvGroup;
  const long long total = static_cast<long long>(n) * h * groups;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    int f, r, x0;
    yuv_item(idx, groups, h, f, r, x0);
    const long long fo = f * p.frame_stride;
    const uint16_t* y = p.y + fo + static_cast<long long>(r) * p.y_pitch + x0;
    const long long co = fo + static_cast<long long>(r) * p.c_pitch + (x0 >> 1) * p.c_step;
    const uint16_t* u = p.u + co;
    const uint16_t* v = p.v + co;
    uint16_t* o = bgr + ((static_cast<long long>(f) * h + r) * w + x0) * 3;
    if (x0 + kYuvGroup <= w) {
      uint32_t yw[4], uw[2], vw[2];
      load_bytes<16>(as_bytes(y), yw);
      if (p.c_step == 1) {
        load_bytes<8>(as_bytes(u), uw);
        load_bytes<8>(as_bytes(v), vw);
      } else {                                     // p210: U0 V0 U1 V1 U2 V2 U3 V3, 16 bits each
        uint32_t uv[4];
        load_bytes<16>(as_bytes(u), uv);
        uw[0] = __byte_perm(uv[0], uv[1], 0x5410); uw[1] = __byte_perm(uv[2], uv[3], 0x5410);
        vw[0] = __byte_perm(uv[0], uv[1], 0x7632); vw[1] = __byte_perm(uv[2], uv[3], 0x7632);
      }
      typename Map::Chroma c[kYuvGroup / 2];
#pragma unroll
      for (int k = 0; k < kYuvGroup / 2; ++k) c[k] = m.chroma(sample10(half_at(uw, k), p.msb), sample10(half_at(vw, k), p.msb));
      uint32_t out[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
      for (int j = 0; j < kYuvGroup; ++j) {
        int B, G, R;
        m.pixel(c[j >> 1], sample10(half_at(yw, j), p.msb), B, G, R);
        put_half(out, 3 * j, B); put_half(out, 3 * j + 1, G); put_half(out, 3 * j + 2, R);
      }
      store_bytes<48>(as_bytes(o), out);
    } else {
      for (int j = 0; x0 + j < w; j += 2) {
        const typename Map::Chroma c = m.chroma(sample10(u[(j >> 1) * p.c_step], p.msb), sample10(v[(j >> 1) * p.c_step], p.msb));
#pragma unroll
        for (int d = 0; d < 2; ++d) {
          int B, G, R;
          m.pixel(c, sample10(y[j + d], p.msb), B, G, R);
          o[3 * (j + d)] = B; o[3 * (j + d) + 1] = G; o[3 * (j + d) + 2] = R;
        }
      }
    }
  }
}

template <class Map>
__global__ void __launch_bounds__(256) yuv422_10_to_bgr48_kernel(const Yuv420Planes16 p, int n, int h, int w, uint16_t* __restrict__ bgr) {
  yuv422_10_to_bgr48_body(p, n, h, w, bgr, Map{});
}

template <class Map>
__device__ __forceinline__ void bgr48_to_yuv422_10_body(const uint16_t* __restrict__ bgr, int n, int h, int w, const Yuv420Planes16& p,
                                                        const Map& m) {
  const int groups = (w + kYuvGroup - 1) / kYuvGroup;
  const long long total = static_cast<long long>(n) * h * groups;
  const int sh = p.msb ? 6 : 0;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    int f, r, x0;
    yuv_item(idx, groups, h, f, r, x0);
    const long long fo = f * p.frame_stride;
    uint16_t* y = p.y + fo + static_cast<long long>(r) * p.y_pitch + x0;
    const long long co = fo + static_cast<long long>(r) * p.c_pitch + (x0 >> 1) * p.c_step;
    uint16_t* u = p.u + co;
    uint16_t* v = p.v + co;
    const uint16_t* in = bgr + ((static_cast<long long>(f) * h + r) * w + x0) * 3;
    if (x0 + kYuvGroup <= w) {
      uint32_t ia[12];
      load_bytes<48>(as_bytes(in), ia);
      uint32_t yw[4] = {0, 0, 0, 0}, uw[2] = {0, 0}, vw[2] = {0, 0};
#pragma unroll
      for (int j = 0; j < kYuvGroup; ++j) {
        const int B = half_at(ia, 3 * j), G = half_at(ia, 3 * j + 1), R = half_at(ia, 3 * j + 2);
        put_half(yw, j, m.y(R, G, B) << sh);
        if ((j & 1) == 0) {                        // the left pixel of its pair
          put_half(uw, j >> 1, m.u(R, G, B) << sh);
          put_half(vw, j >> 1, m.v(R, G, B) << sh);
        }
      }
      store_bytes<16>(as_bytes(y), yw);
      if (p.c_step == 1) {
        store_bytes<8>(as_bytes(u), uw);
        store_bytes<8>(as_bytes(v), vw);
      } else {
        const uint32_t uv[4] = {__byte_perm(uw[0], vw[0], 0x5410), __byte_perm(uw[0], vw[0], 0x7632),
                                __byte_perm(uw[1], vw[1], 0x5410), __byte_perm(uw[1], vw[1], 0x7632)};
        store_bytes<16>(as_bytes(u), uv);
      }
    } else {
      for (int j = 0; x0 + j < w; j += 2) {
        const uint16_t* a = in + 3 * j;
        u[(j >> 1) * p.c_step] = static_cast<uint16_t>(m.u(a[2], a[1], a[0]) << sh);
        v[(j >> 1) * p.c_step] = static_cast<uint16_t>(m.v(a[2], a[1], a[0]) << sh);
#pragma unroll
        for (int d = 0; d < 2; ++d) {
          const uint16_t* q = in + 3 * (j + d);
          y[j + d] = static_cast<uint16_t>(m.y(q[2], q[1], q[0]) << sh);
        }
      }
    }
  }
}

template <class Map>
__global__ void __launch_bounds__(256) bgr48_to_yuv422_10_kernel(const uint16_t* __restrict__ bgr, int n, int h, int w, const Yuv420Planes16 p) {
  bgr48_to_yuv422_10_body(bgr, n, h, w, p, Map{});
}

// The checks the conversion entry points make before any launch (pitches in bytes for 8-bit planes, in elements for 16-bit ones).
static int check_yuv420(const char* fn, int n, int h, int w, int y_pitch, int c_pitch, int c_step, long long frame_stride,
                        bool deep = false) {
  SAVSR_REQUIRE(n >= 0 && h > 0 && w > 0, "%s: bad shape n=%d h=%d w=%d", fn, n, h, w);
  SAVSR_REQUIRE(h % 2 == 0 && w % 2 == 0, "%s: YUV 4:2:0 needs an even frame size, got %dx%d", fn, h, w);
  SAVSR_REQUIRE(c_step == 1 || c_step == 2, "%s: c_step must be 1 (%s) or 2 (%s), got %d", fn, deep ? "yuv420p10le" : "yuv420p",
                deep ? "p010" : "nv12", c_step);
  SAVSR_REQUIRE(y_pitch >= w, "%s: y_pitch %d < width %d", fn, y_pitch, w);
  SAVSR_REQUIRE(c_pitch >= c_step * (w / 2), "%s: c_pitch %d < chroma row of %d %s", fn, c_pitch, c_step * (w / 2),
                deep ? "elements" : "bytes");
  SAVSR_REQUIRE(frame_stride >= 0, "%s: negative frame_stride %lld", fn, frame_stride);
  return 0;
}

static unsigned grid_for(const savsr_ctx* ctx, long long items) {
  const long long b = (items + 255) / 256, cap = 16LL * ctx->sm_count;
  return static_cast<unsigned>(b < cap ? b : cap);
}

static unsigned yuv_blocks(const savsr_ctx* ctx, int n, int h, int w) {
  return grid_for(ctx, static_cast<long long>(n) * (h / 2) * ((w + kYuvGroup - 1) / kYuvGroup));
}

// The kernel of (colorspace, range) for the _cs entry points: the cv2-exact kernel of the plain entry point for (BT601, TV), else the
// pair's H.273 instantiation; an error naming the value for anything not in enum savsr_colorspace / savsr_color_range.
template <class F>
static int cs_kernel(const char* fn, int colorspace, int range, F plain, const F (&table)[3][2], F* k) {
  SAVSR_REQUIRE(colorspace >= SAVSR_COLORSPACE_BT601 && colorspace <= SAVSR_COLORSPACE_BT2020NC,
                "%s: unknown colorspace %d (0 BT601, 1 BT709, 2 BT2020NC)", fn, colorspace);
  SAVSR_REQUIRE(range == SAVSR_RANGE_TV || range == SAVSR_RANGE_PC, "%s: unknown color range %d (0 TV, 1 PC)", fn, range);
  *k = colorspace == SAVSR_COLORSPACE_BT601 && range == SAVSR_RANGE_TV ? plain : table[colorspace][range];
  return 0;
}
#define SAVSR_CS_TABLE(kernel) {{nullptr, kernel<0, 1>}, {kernel<1, 0>, kernel<1, 1>}, {kernel<2, 0>, kernel<2, 1>}}
using Dec8Kernel = void (*)(const Yuv420Planes, int, int, int, uint8_t*);
using Enc8Kernel = void (*)(const uint8_t*, int, int, int, const Yuv420Planes);
using Dec10Kernel = void (*)(const Yuv420Planes16, int, int, int, uint16_t*);
using Enc10Kernel = void (*)(const uint16_t*, int, int, int, const Yuv420Planes16);
static const Dec8Kernel kDec8Cs[3][2] = SAVSR_CS_TABLE(yuv420_to_bgr_cs_kernel);
static const Enc8Kernel kEnc8Cs[3][2] = SAVSR_CS_TABLE(bgr_to_yuv420_cs_kernel);
static const Dec10Kernel kDec10Cs[3][2] = SAVSR_CS_TABLE(yuv420_10_to_bgr48_cs_kernel);
static const Enc10Kernel kEnc10Cs[3][2] = SAVSR_CS_TABLE(bgr48_to_yuv420_10_cs_kernel);
#undef SAVSR_CS_TABLE

// The four conversions, with the kernel to launch.
static int yuv420_to_bgr(const char* fn, savsr_ctx* ctx, const uint8_t* y, int y_pitch, const uint8_t* u, const uint8_t* v, int c_pitch,
                         int c_step, int64_t frame_stride, int n, int h, int w, uint8_t* bgr, Dec8Kernel k, savsr_stream st) {
  SAVSR_REQUIRE(ctx && y && u && v && bgr, "%s: null pointer", fn);
  if (check_yuv420(fn, n, h, w, y_pitch, c_pitch, c_step, frame_stride)) return 1;
  if (n == 0) return 0;
  DeviceGuard guard(ctx->device);
  const Yuv420Planes p{const_cast<uint8_t*>(y), const_cast<uint8_t*>(u), const_cast<uint8_t*>(v), y_pitch, c_pitch, c_step, frame_stride};
  k<<<yuv_blocks(ctx, n, h, w), 256, 0, static_cast<cudaStream_t>(st)>>>(p, n, h, w, bgr);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

static int bgr_to_yuv420(const char* fn, savsr_ctx* ctx, const uint8_t* bgr, int n, int h, int w, uint8_t* y, int y_pitch, uint8_t* u,
                         uint8_t* v, int c_pitch, int c_step, int64_t frame_stride, Enc8Kernel k, savsr_stream st) {
  SAVSR_REQUIRE(ctx && bgr && y && u && v, "%s: null pointer", fn);
  if (check_yuv420(fn, n, h, w, y_pitch, c_pitch, c_step, frame_stride)) return 1;
  if (n == 0) return 0;
  DeviceGuard guard(ctx->device);
  const Yuv420Planes p{y, u, v, y_pitch, c_pitch, c_step, frame_stride};
  k<<<yuv_blocks(ctx, n, h, w), 256, 0, static_cast<cudaStream_t>(st)>>>(bgr, n, h, w, p);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

static int yuv420_10_to_bgr48(const char* fn, savsr_ctx* ctx, const uint16_t* y, int y_pitch, const uint16_t* u, const uint16_t* v,
                              int c_pitch, int c_step, int64_t frame_stride, int msb, int n, int h, int w, uint16_t* bgr, Dec10Kernel k,
                              savsr_stream st) {
  SAVSR_REQUIRE(ctx && y && u && v && bgr, "%s: null pointer", fn);
  if (check_yuv420(fn, n, h, w, y_pitch, c_pitch, c_step, frame_stride, true)) return 1;
  SAVSR_REQUIRE(msb == 0 || msb == 1, "%s: msb must be 0 (yuv420p10le) or 1 (p010), got %d", fn, msb);
  if (n == 0) return 0;
  DeviceGuard guard(ctx->device);
  const Yuv420Planes16 p{const_cast<uint16_t*>(y), const_cast<uint16_t*>(u), const_cast<uint16_t*>(v), y_pitch, c_pitch, c_step,
                         frame_stride, msb};
  k<<<yuv_blocks(ctx, n, h, w), 256, 0, static_cast<cudaStream_t>(st)>>>(p, n, h, w, bgr);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

static int bgr48_to_yuv420_10(const char* fn, savsr_ctx* ctx, const uint16_t* bgr, int n, int h, int w, uint16_t* y, int y_pitch,
                              uint16_t* u, uint16_t* v, int c_pitch, int c_step, int64_t frame_stride, int msb, Enc10Kernel k,
                              savsr_stream st) {
  SAVSR_REQUIRE(ctx && bgr && y && u && v, "%s: null pointer", fn);
  if (check_yuv420(fn, n, h, w, y_pitch, c_pitch, c_step, frame_stride, true)) return 1;
  SAVSR_REQUIRE(msb == 0 || msb == 1, "%s: msb must be 0 (yuv420p10le) or 1 (p010), got %d", fn, msb);
  if (n == 0) return 0;
  DeviceGuard guard(ctx->device);
  const Yuv420Planes16 p{y, u, v, y_pitch, c_pitch, c_step, frame_stride, msb};
  k<<<yuv_blocks(ctx, n, h, w), 256, 0, static_cast<cudaStream_t>(st)>>>(bgr, n, h, w, p);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

// The 4:2:2 kernels of each (colorspace, range): [BT601][TV] is the cv2-exact map, the others their H.273 maps.
#define SAVSR_422_TABLE(kernel, M)                                                                        \
  {{kernel<Cv2Map##M>, kernel<CsMap##M<0, 1>>}, {kernel<CsMap##M<1, 0>>, kernel<CsMap##M<1, 1>>}, \
   {kernel<CsMap##M<2, 0>>, kernel<CsMap##M<2, 1>>}}
using Dec422Kernel = void (*)(const Yuv422Planes, int, int, int, uint8_t*);
using Enc422Kernel = void (*)(const uint8_t*, int, int, int, const Yuv422Planes);
static const Dec422Kernel kDec422[3][2] = SAVSR_422_TABLE(yuv422_to_bgr_kernel, 8);
static const Enc422Kernel kEnc422[3][2] = SAVSR_422_TABLE(bgr_to_yuv422_kernel, 8);
static const Dec10Kernel kDec422_10[3][2] = SAVSR_422_TABLE(yuv422_10_to_bgr48_kernel, 10);
static const Enc10Kernel kEnc422_10[3][2] = SAVSR_422_TABLE(bgr48_to_yuv422_10_kernel, 10);
#undef SAVSR_422_TABLE

// The checks of the 4:2:2 entry points before any launch; T is the sample type (pitches and strides in its elements).
template <class T>
static int check_yuv422(const char* fn, int n, int h, int w, const T* y, int y_pitch, int y_step, const T* u, const T* v, int c_pitch,
                        int c_step, long long frame_stride) {
  constexpr bool deep = sizeof(T) == 2;
  SAVSR_REQUIRE(n >= 0 && h > 0 && w > 0, "%s: bad shape n=%d h=%d w=%d", fn, n, h, w);
  SAVSR_REQUIRE(w % 2 == 0, "%s: YUV 4:2:2 needs an even width, got %dx%d", fn, h, w);
  if (deep) {
    SAVSR_REQUIRE(y_step == 1 && (c_step == 1 || c_step == 2),
                  "%s: (y_step, c_step) must be (1, 1) (yuv422p10le) or (1, 2) (p210), got (%d, %d)", fn, y_step, c_step);
  } else {
    SAVSR_REQUIRE((y_step == 1 && (c_step == 1 || c_step == 2)) || (y_step == 2 && c_step == 4),
                  "%s: (y_step, c_step) must be (1, 1) (yuv422p), (1, 2) (nv16) or (2, 4) (yuyv422, uyvy422), got (%d, %d)", fn, y_step,
                  c_step);
  }
  SAVSR_REQUIRE(y_pitch >= y_step * w, "%s: y_pitch %d < row of %d %s", fn, y_pitch, y_step * w, deep ? "elements" : "bytes");
  SAVSR_REQUIRE(c_pitch >= c_step * (w / 2), "%s: c_pitch %d < chroma row of %d %s", fn, c_pitch, c_step * (w / 2),
                deep ? "elements" : "bytes");
  SAVSR_REQUIRE(c_step != 2 || v == u + 1, "%s: interleaved chroma (c_step 2) needs v = u + 1", fn);
  SAVSR_REQUIRE(y_step != 2 || (c_pitch == y_pitch && ((u == y + 1 && v == y + 3) || (u == y - 1 && v == y + 1))),
                "%s: packed 4:2:2 needs c_pitch = y_pitch and yuyv422 (u = y + 1, v = y + 3) or uyvy422 (u = y - 1, v = y + 1)", fn);
  SAVSR_REQUIRE(frame_stride >= 0, "%s: negative frame_stride %lld", fn, frame_stride);
  return 0;
}

static unsigned yuv422_blocks(const savsr_ctx* ctx, int n, int h, int w) {
  return grid_for(ctx, static_cast<long long>(n) * h * ((w + kYuvGroup - 1) / kYuvGroup));
}

}  // namespace savsr

using namespace savsr;

extern "C" int savsr_yuv420_to_bgr(savsr_ctx* ctx, const uint8_t* y, int y_pitch, const uint8_t* u, const uint8_t* v, int c_pitch,
                                   int c_step, int64_t frame_stride, int n, int h, int w, uint8_t* bgr, savsr_stream st) {
  return savsr::yuv420_to_bgr("savsr_yuv420_to_bgr", ctx, y, y_pitch, u, v, c_pitch, c_step, frame_stride, n, h, w, bgr, yuv420_to_bgr_kernel, st);
}

extern "C" int savsr_yuv420_to_bgr_cs(savsr_ctx* ctx, const uint8_t* y, int y_pitch, const uint8_t* u, const uint8_t* v, int c_pitch,
                                      int c_step, int64_t frame_stride, int n, int h, int w, uint8_t* bgr, int colorspace, int range,
                                      savsr_stream st) {
  const char* fn = "savsr_yuv420_to_bgr_cs";
  Dec8Kernel k;
  if (cs_kernel(fn, colorspace, range, static_cast<Dec8Kernel>(yuv420_to_bgr_kernel), kDec8Cs, &k)) return 1;
  return savsr::yuv420_to_bgr(fn, ctx, y, y_pitch, u, v, c_pitch, c_step, frame_stride, n, h, w, bgr, k, st);
}

extern "C" int savsr_bgr_to_yuv420(savsr_ctx* ctx, const uint8_t* bgr, int n, int h, int w, uint8_t* y, int y_pitch, uint8_t* u, uint8_t* v,
                                   int c_pitch, int c_step, int64_t frame_stride, savsr_stream st) {
  return savsr::bgr_to_yuv420("savsr_bgr_to_yuv420", ctx, bgr, n, h, w, y, y_pitch, u, v, c_pitch, c_step, frame_stride, bgr_to_yuv420_kernel, st);
}

extern "C" int savsr_bgr_to_yuv420_cs(savsr_ctx* ctx, const uint8_t* bgr, int n, int h, int w, uint8_t* y, int y_pitch, uint8_t* u,
                                      uint8_t* v, int c_pitch, int c_step, int64_t frame_stride, int colorspace, int range, savsr_stream st) {
  const char* fn = "savsr_bgr_to_yuv420_cs";
  Enc8Kernel k;
  if (cs_kernel(fn, colorspace, range, static_cast<Enc8Kernel>(bgr_to_yuv420_kernel), kEnc8Cs, &k)) return 1;
  return savsr::bgr_to_yuv420(fn, ctx, bgr, n, h, w, y, y_pitch, u, v, c_pitch, c_step, frame_stride, k, st);
}

extern "C" int savsr_yuv420_10_to_bgr48(savsr_ctx* ctx, const uint16_t* y, int y_pitch, const uint16_t* u, const uint16_t* v, int c_pitch,
                                        int c_step, int64_t frame_stride, int msb, int n, int h, int w, uint16_t* bgr, savsr_stream st) {
  return savsr::yuv420_10_to_bgr48("savsr_yuv420_10_to_bgr48", ctx, y, y_pitch, u, v, c_pitch, c_step, frame_stride, msb, n, h, w, bgr,
                                   yuv420_10_to_bgr48_kernel, st);
}

extern "C" int savsr_yuv420_10_to_bgr48_cs(savsr_ctx* ctx, const uint16_t* y, int y_pitch, const uint16_t* u, const uint16_t* v,
                                           int c_pitch, int c_step, int64_t frame_stride, int msb, int n, int h, int w, uint16_t* bgr,
                                           int colorspace, int range, savsr_stream st) {
  const char* fn = "savsr_yuv420_10_to_bgr48_cs";
  Dec10Kernel k;
  if (cs_kernel(fn, colorspace, range, static_cast<Dec10Kernel>(yuv420_10_to_bgr48_kernel), kDec10Cs, &k)) return 1;
  return savsr::yuv420_10_to_bgr48(fn, ctx, y, y_pitch, u, v, c_pitch, c_step, frame_stride, msb, n, h, w, bgr, k, st);
}

extern "C" int savsr_bgr48_to_yuv420_10(savsr_ctx* ctx, const uint16_t* bgr, int n, int h, int w, uint16_t* y, int y_pitch, uint16_t* u,
                                        uint16_t* v, int c_pitch, int c_step, int64_t frame_stride, int msb, savsr_stream st) {
  return savsr::bgr48_to_yuv420_10("savsr_bgr48_to_yuv420_10", ctx, bgr, n, h, w, y, y_pitch, u, v, c_pitch, c_step, frame_stride, msb,
                                   bgr48_to_yuv420_10_kernel, st);
}

extern "C" int savsr_bgr48_to_yuv420_10_cs(savsr_ctx* ctx, const uint16_t* bgr, int n, int h, int w, uint16_t* y, int y_pitch, uint16_t* u,
                                           uint16_t* v, int c_pitch, int c_step, int64_t frame_stride, int msb, int colorspace, int range,
                                           savsr_stream st) {
  const char* fn = "savsr_bgr48_to_yuv420_10_cs";
  Enc10Kernel k;
  if (cs_kernel(fn, colorspace, range, static_cast<Enc10Kernel>(bgr48_to_yuv420_10_kernel), kEnc10Cs, &k)) return 1;
  return savsr::bgr48_to_yuv420_10(fn, ctx, bgr, n, h, w, y, y_pitch, u, v, c_pitch, c_step, frame_stride, msb, k, st);
}

extern "C" int savsr_yuv422_to_bgr_cs(savsr_ctx* ctx, const uint8_t* y, int y_pitch, int y_step, const uint8_t* u, const uint8_t* v,
                                      int c_pitch, int c_step, int64_t frame_stride, int n, int h, int w, uint8_t* bgr, int colorspace,
                                      int range, savsr_stream st) {
  const char* fn = "savsr_yuv422_to_bgr_cs";
  Dec422Kernel k;
  if (cs_kernel(fn, colorspace, range, kDec422[0][0], kDec422, &k)) return 1;
  SAVSR_REQUIRE(ctx && y && u && v && bgr, "%s: null pointer", fn);
  if (check_yuv422(fn, n, h, w, y, y_pitch, y_step, u, v, c_pitch, c_step, frame_stride)) return 1;
  if (n == 0) return 0;
  DeviceGuard guard(ctx->device);
  const Yuv422Planes p{const_cast<uint8_t*>(y), const_cast<uint8_t*>(u), const_cast<uint8_t*>(v), y_pitch, y_step, c_pitch, c_step,
                       frame_stride};
  k<<<yuv422_blocks(ctx, n, h, w), 256, 0, static_cast<cudaStream_t>(st)>>>(p, n, h, w, bgr);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int savsr_bgr_to_yuv422_cs(savsr_ctx* ctx, const uint8_t* bgr, int n, int h, int w, uint8_t* y, int y_pitch, int y_step,
                                      uint8_t* u, uint8_t* v, int c_pitch, int c_step, int64_t frame_stride, int colorspace, int range,
                                      savsr_stream st) {
  const char* fn = "savsr_bgr_to_yuv422_cs";
  Enc422Kernel k;
  if (cs_kernel(fn, colorspace, range, kEnc422[0][0], kEnc422, &k)) return 1;
  SAVSR_REQUIRE(ctx && bgr && y && u && v, "%s: null pointer", fn);
  if (check_yuv422<uint8_t>(fn, n, h, w, y, y_pitch, y_step, u, v, c_pitch, c_step, frame_stride)) return 1;
  if (n == 0) return 0;
  DeviceGuard guard(ctx->device);
  const Yuv422Planes p{y, u, v, y_pitch, y_step, c_pitch, c_step, frame_stride};
  k<<<yuv422_blocks(ctx, n, h, w), 256, 0, static_cast<cudaStream_t>(st)>>>(bgr, n, h, w, p);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int savsr_yuv422_10_to_bgr48_cs(savsr_ctx* ctx, const uint16_t* y, int y_pitch, int y_step, const uint16_t* u, const uint16_t* v,
                                           int c_pitch, int c_step, int64_t frame_stride, int msb, int n, int h, int w, uint16_t* bgr,
                                           int colorspace, int range, savsr_stream st) {
  const char* fn = "savsr_yuv422_10_to_bgr48_cs";
  Dec10Kernel k;
  if (cs_kernel(fn, colorspace, range, kDec422_10[0][0], kDec422_10, &k)) return 1;
  SAVSR_REQUIRE(ctx && y && u && v && bgr, "%s: null pointer", fn);
  if (check_yuv422(fn, n, h, w, y, y_pitch, y_step, u, v, c_pitch, c_step, frame_stride)) return 1;
  SAVSR_REQUIRE(msb == 0 || msb == 1, "%s: msb must be 0 (yuv422p10le) or 1 (p210), got %d", fn, msb);
  if (n == 0) return 0;
  DeviceGuard guard(ctx->device);
  const Yuv420Planes16 p{const_cast<uint16_t*>(y), const_cast<uint16_t*>(u), const_cast<uint16_t*>(v), y_pitch, c_pitch, c_step,
                         frame_stride, msb};
  k<<<yuv422_blocks(ctx, n, h, w), 256, 0, static_cast<cudaStream_t>(st)>>>(p, n, h, w, bgr);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int savsr_bgr48_to_yuv422_10_cs(savsr_ctx* ctx, const uint16_t* bgr, int n, int h, int w, uint16_t* y, int y_pitch, int y_step,
                                           uint16_t* u, uint16_t* v, int c_pitch, int c_step, int64_t frame_stride, int msb,
                                           int colorspace, int range, savsr_stream st) {
  const char* fn = "savsr_bgr48_to_yuv422_10_cs";
  Enc10Kernel k;
  if (cs_kernel(fn, colorspace, range, kEnc422_10[0][0], kEnc422_10, &k)) return 1;
  SAVSR_REQUIRE(ctx && bgr && y && u && v, "%s: null pointer", fn);
  if (check_yuv422<uint16_t>(fn, n, h, w, y, y_pitch, y_step, u, v, c_pitch, c_step, frame_stride)) return 1;
  SAVSR_REQUIRE(msb == 0 || msb == 1, "%s: msb must be 0 (yuv422p10le) or 1 (p210), got %d", fn, msb);
  if (n == 0) return 0;
  DeviceGuard guard(ctx->device);
  const Yuv420Planes16 p{y, u, v, y_pitch, c_pitch, c_step, frame_stride, msb};
  k<<<yuv422_blocks(ctx, n, h, w), 256, 0, static_cast<cudaStream_t>(st)>>>(bgr, n, h, w, p);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int savsr_widen_u8_to_u16(savsr_ctx* ctx, const uint8_t* src, int n, int h, int w, uint16_t* dst, savsr_stream st) {
  SAVSR_REQUIRE(ctx && src && dst, "savsr_widen_u8_to_u16: null pointer");
  SAVSR_REQUIRE(n >= 0 && h > 0 && w > 0, "savsr_widen_u8_to_u16: bad shape n=%d h=%d w=%d", n, h, w);
  if (n == 0) return 0;
  DeviceGuard guard(ctx->device);
  const long long count = static_cast<long long>(n) * h * w * 3;
  widen_u8_to_u16_kernel<<<grid_for(ctx, (count + 15) / 16), 256, 0, static_cast<cudaStream_t>(st)>>>(src, dst, count);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}
