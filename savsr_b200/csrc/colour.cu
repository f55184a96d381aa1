// YUV <-> packed BGR on the device, so decoded video (NVDEC NV12 / P010 surfaces, ffmpeg rawvideo pipes) enters the forward and its HR
// frames leave for an encoder without a colour conversion on the CPU.  One decode and one encode kernel template cover every layout,
// subsampling, depth and colour pair.
//
// Plane model (both directions, every layout): frame k's planes are frame 0's plus k * frame_stride.  Frame row r's Y samples start at
// y + r * y_pitch, y_step apart; chroma row c's U and V samples start at u + c * c_pitch and v + c * c_pitch, c_step apart.  Pitches and
// strides count samples: bytes for 8-bit planes, uint16 elements for 10-bit ones.  The layouts:
//   planar (yuv420p, yuv422p, yuv420p10le, yuv422p10le): separate U and V planes; y_step 1, c_step 1;
//   semi-planar (nv12, nv16, p010, p210): one plane of interleaved U, V samples, v = u + 1; y_step 1, c_step 2;
//   packed 4:2:2 (yuyv422, uyvy422; 8-bit only): y, u and v point into the same rows of 4-byte macropixels; y_step 2, c_step 4,
//   c_pitch = y_pitch; yuyv422 is Y0 U0 Y1 V0 (u = y + 1, v = y + 3), uyvy422 U0 Y0 V0 Y1 (u = y - 1, v = y + 1).
// The BGR side is contiguous [n][h][w][3].
//
// Subsampling: ROWS frame rows share one chroma row, 2 for 4:2:0 and 1 for 4:2:2, and each horizontal pixel pair shares one (U, V).
// Decoding gives every pixel its pair's chroma: cv2's COLOR_YUV2BGR_I420 / _NV12 / _YUYV / _UYVY.  Encoding takes U and V from the left
// pixel of the pair in the first of the ROWS rows: the top-left of a 2x2 block in 4:2:0 (cv2's COLOR_BGR2YUV_I420, no averaging), the
// co-sited position of H.264, HEVC and ProRes 4:2:2 in 4:2:2.  So a 4:2:0 encode is the 4:2:2 encode with its odd chroma rows dropped.
// (cv2's COLOR_BGR2YUV_YUYV averages the pair's chroma and rounds Y otherwise: it is not this.)
//
// Work split: a thread owns 8 pixels (four chroma pairs) of each of its ROWS rows, so every chroma sample is read or written once and
// odd 4:2:2 heights need nothing special.  It issues the loads of all its rows before it converts any, and moves each row with the widest
// accesses the row's alignment allows (all rows of one frame share it; see load_bytes / store_bytes).  A row's last group may be
// narrower (w % 8): it takes the sample-wise path.  The kernels move bytes and do a few integer multiplies per pixel: bound by HBM.
//
// Pixel maps: Cv2Map8 is byte-exact with OpenCV 4's cv::cvtColor, BT.601 limited range in 20-bit fixed point (constants in common.cuh).
// 10-bit YUV <-> 16-bit BGR (Cv2Map10) uses the same matrix and chroma handling in fixed-point forms rescaled to the deeper samples; the
// 10 bits sit in bits 0-9 of their uint16 (yuv420p10le, yuv422p10le: msb 0) or in bits 6-15 (p010, p210: msb 1).  A thread's rows are
// 16 bytes of Y and 48 of BGR there, so 16-byte accesses are used where the row's alignment allows.  The other (colorspace, range) pairs
// (the _cs entry points) use that pair's H.273 map, CsMap8 / CsMap10, one instantiation per pair with the coefficients of kYuvCoeffs8 /
// kYuvCoeffs10 as compile-time constants.  widen_u8_to_u16 brings 8-bit BGR frames into a 16-bit ring.
#include <type_traits>

#include "common.cuh"

namespace savsr {

constexpr int kYuvGroup = 8;   // pixels per thread and row: four chroma pairs

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

template <class T>
__device__ __forceinline__ const uint8_t* as_bytes(const T* p) { return reinterpret_cast<const uint8_t*>(p); }
template <class T>
__device__ __forceinline__ uint8_t* as_bytes(T* p) { return reinterpret_cast<uint8_t*>(p); }

__device__ __forceinline__ int sat_u8(int v) { return min(max(v, 0), 255); }
__device__ __forceinline__ int sat_u10(int v) { return min(max(v, 0), 1023); }
__device__ __forceinline__ int sat_u16(int v) { return min(max(v, 0), 65535); }

// The kernels are written over a pixel map: chroma(U, V) once per chroma pair and pixel(c, Y, B, G, R) per pixel (decode), and
// y, u, v of (R, G, B) (encode).  Cv2Map8: OpenCV's BT.601 limited-range fixed point.  Encoding lies in [16, 235] (Y) and [16, 240]
// (U, V) for every 8-bit input, so it needs no saturation.
struct Cv2Map8 {
  struct Chroma { int r, g, b; };
  __device__ __forceinline__ Chroma chroma(int U, int V) const {
    const int u = U - 128, v = V - 128;
    return {kYuvHalf + kYuvVR * v, kYuvHalf + kYuvVG * v + kYuvUG * u, kYuvHalf + kYuvUB * u};
  }
  __device__ __forceinline__ void pixel(const Chroma& c, int Y, int& B, int& G, int& R) const {
    const int y = max(Y - 16, 0) * kYuvY;
    B = sat_u8((y + c.b) >> kYuvShift);
    G = sat_u8((y + c.g) >> kYuvShift);
    R = sat_u8((y + c.r) >> kYuvShift);
  }
  __device__ __forceinline__ int y(int R, int G, int B) const { return (kRgbYR * R + kRgbYG * G + kRgbYB * B + (16 << kYuvShift) + kYuvHalf) >> kYuvShift; }
  __device__ __forceinline__ int u(int R, int G, int B) const { return (kRgbUR * R + kRgbUG * G + kRgbUB * B + (128 << kYuvShift) + kYuvHalf) >> kYuvShift; }
  __device__ __forceinline__ int v(int R, int G, int B) const { return (kRgbVR * R + kRgbVG * G + kRgbVB * B + (128 << kYuvShift) + kYuvHalf) >> kYuvShift; }
};

// CsMap8<CS, RNG>: the H.273 map of one (matrix, range) pair, its coefficients compile-time constants from kYuvCoeffs8 (one
// instantiation per pair: with the coefficients passed by value instead, the 8-bit encode needed 62 registers instead of 40 and ran
// 17 % slower at 1080p x 26).
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

// The 10-bit pixel maps, as Cv2Map8 / CsMap8 (10-bit YUV samples, 16-bit BGR; coefficients from common.cuh and kYuvCoeffs10).
struct Cv2Map10 {
  struct Chroma { long long r, g, b; };
  __device__ __forceinline__ Chroma chroma(int U, int V) const {
    const int u = U - 512, v = V - 512;
    return {kYuv10Half + static_cast<long long>(kYuv10VR) * v,
            kYuv10Half + static_cast<long long>(kYuv10VG) * v + static_cast<long long>(kYuv10UG) * u,
            kYuv10Half + static_cast<long long>(kYuv10UB) * u};
  }
  __device__ __forceinline__ void pixel(const Chroma& c, int Y, int& B, int& G, int& R) const {
    const long long y = static_cast<long long>(max(Y - 64, 0)) * kYuv10Y;
    B = sat_u16(static_cast<int>((y + c.b) >> kYuv10Shift));
    G = sat_u16(static_cast<int>((y + c.g) >> kYuv10Shift));
    R = sat_u16(static_cast<int>((y + c.r) >> kYuv10Shift));
  }
  __device__ __forceinline__ int y(int R, int G, int B) const {
    return (kRgb10YR * R + kRgb10YG * G + kRgb10YB * B + (64 << kRgb10Shift) + kRgb10Half) >> kRgb10Shift;
  }
  __device__ __forceinline__ int u(int R, int G, int B) const {
    return (kRgb10UR * R + kRgb10UG * G + kRgb10UB * B + (512 << kRgb10Shift) + kRgb10Half) >> kRgb10Shift;
  }
  __device__ __forceinline__ int v(int R, int G, int B) const {
    return (kRgb10VR * R + kRgb10VG * G + kRgb10VB * B + (512 << kRgb10Shift) + kRgb10Half) >> kRgb10Shift;
  }
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

// The cv2-exact map and the H.273 maps of the sample type T.
template <class T>
using Cv2Map = std::conditional_t<sizeof(T) == 1, Cv2Map8, Cv2Map10>;
template <class T, int CS, int RNG>
using CsMap = std::conditional_t<sizeof(T) == 1, CsMap8<CS, RNG>, CsMap10<CS, RNG>>;

// The planes of n frames, as the header comment describes them.  msb: where a 16-bit sample keeps its 10 bits (unused for 8 bits).
// y_step comes last: see the register note above yuv_to_bgr_kernel.
template <class T>
struct YuvPlanes {
  T* y;
  T* u;
  T* v;
  int y_pitch, c_pitch, c_step;
  long long frame_stride;
  int msb, y_step;
};

// What depends on the sample type T: 8-bit samples packed four to a 32-bit word, 16-bit ones two.
template <class T>
struct Samples {
  static constexpr int kBits = 8 * sizeof(T), kPerWord = 4 / sizeof(T);
  static constexpr int kRow = kYuvGroup / kPerWord;   // words of a thread's Y samples of one row
  static constexpr int kChroma = kRow / 2;            // words of its U (or V) samples
  // __byte_perm selectors: the U and V words of interleaved U, V words (split), and the interleaved low and high words (join).
  static constexpr unsigned kSplitU = sizeof(T) == 1 ? 0x6420 : 0x5410, kSplitV = sizeof(T) == 1 ? 0x7531 : 0x7632;
  static constexpr unsigned kJoinLo = sizeof(T) == 1 ? 0x5140 : 0x5410, kJoinHi = sizeof(T) == 1 ? 0x7362 : 0x7632;

  template <int N>
  static __device__ __forceinline__ int at(const uint32_t (&w)[N], int i) {
    return (w[i / kPerWord] >> (kBits * (i % kPerWord))) & ((1u << kBits) - 1);
  }
  template <int N>
  static __device__ __forceinline__ void put(uint32_t (&w)[N], int i, int v) { w[i / kPerWord] |= static_cast<uint32_t>(v) << (kBits * (i % kPerWord)); }
  // The value of a stored sample, and the shift that stores a value.
  static __device__ __forceinline__ int value(int s, int msb) {
    if constexpr (sizeof(T) == 1) return s;
    else return msb ? s >> 6 : s & 0x3ff;
  }
  static __device__ __forceinline__ int shift(int msb) { return sizeof(T) == 2 && msb ? 6 : 0; }
};

// A thread's Y words of its ROWS rows (yr: where each starts), then its U and V words, from planar or semi-planar planes; and their store.
template <class T, int ROWS, int R, int C>
__device__ __forceinline__ void load_planar(const T* const (&yr)[ROWS], const T* u, const T* v, int c_step, uint32_t (&yw)[ROWS][R],
                                            uint32_t (&uw)[C], uint32_t (&vw)[C]) {
#pragma unroll
  for (int r = 0; r < ROWS; ++r) load_bytes<4 * R>(as_bytes(yr[r]), yw[r]);
  if (c_step == 1) {
    load_bytes<4 * C>(as_bytes(u), uw);
    load_bytes<4 * C>(as_bytes(v), vw);
  } else {                                         // U0 V0 U1 V1 U2 V2 U3 V3
    uint32_t uv[2 * C];
    load_bytes<8 * C>(as_bytes(u), uv);
#pragma unroll
    for (int k = 0; k < C; ++k) {
      uw[k] = __byte_perm(uv[2 * k], uv[2 * k + 1], Samples<T>::kSplitU);
      vw[k] = __byte_perm(uv[2 * k], uv[2 * k + 1], Samples<T>::kSplitV);
    }
  }
}

template <class T, int ROWS, int R, int C>
__device__ __forceinline__ void store_planar(T* const (&yr)[ROWS], T* u, T* v, int c_step, const uint32_t (&yw)[ROWS][R], const uint32_t (&uw)[C],
                                             const uint32_t (&vw)[C]) {
  store_bytes<4 * R>(as_bytes(yr[0]), yw[0]);                       // not a loop: see the register note
  if constexpr (ROWS == 2) store_bytes<4 * R>(as_bytes(yr[1]), yw[1]);
  if (c_step == 1) {
    store_bytes<4 * C>(as_bytes(u), uw);
    store_bytes<4 * C>(as_bytes(v), vw);
  } else {
    uint32_t uv[2 * C];
#pragma unroll
    for (int k = 0; k < C; ++k) {
      uv[2 * k] = __byte_perm(uw[k], vw[k], Samples<T>::kJoinLo);
      uv[2 * k + 1] = __byte_perm(uw[k], vw[k], Samples<T>::kJoinHi);
    }
    store_bytes<8 * C>(as_bytes(u), uv);
  }
}

// The same for packed 4:2:2: four macropixels, from or to whichever of y and u comes first.
__device__ __forceinline__ void load_packed(const uint8_t* y, const uint8_t* u, uint32_t (&yw)[2], uint32_t (&uw)[1], uint32_t (&vw)[1]) {
  const bool uyvy = u < y;
  uint32_t q[4];
  load_bytes<16>(uyvy ? u : y, q);
  const unsigned sy = uyvy ? 0x7531 : 0x6420, sc = uyvy ? 0x6420 : 0x7531;
  yw[0] = __byte_perm(q[0], q[1], sy);
  yw[1] = __byte_perm(q[2], q[3], sy);
  const uint32_t c01 = __byte_perm(q[0], q[1], sc), c23 = __byte_perm(q[2], q[3], sc);     // U0 V0 U1 V1, U2 V2 U3 V3
  uw[0] = __byte_perm(c01, c23, 0x6420);
  vw[0] = __byte_perm(c01, c23, 0x7531);
}

__device__ __forceinline__ void store_packed(uint8_t* y, uint8_t* u, const uint32_t (&yw)[2], const uint32_t (&uw)[1], const uint32_t (&vw)[1]) {
  const bool uyvy = u < y;
  const uint32_t c01 = __byte_perm(uw[0], vw[0], 0x5140), c23 = __byte_perm(uw[0], vw[0], 0x7362);   // U0 V0 U1 V1, U2 V2 U3 V3
  const unsigned s0 = uyvy ? 0x1504 : 0x5140, s1 = uyvy ? 0x3726 : 0x7362;
  const uint32_t q[4] = {__byte_perm(yw[0], c01, s0), __byte_perm(yw[0], c01, s1), __byte_perm(yw[1], c23, s0), __byte_perm(yw[1], c23, s1)};
  store_bytes<16>(uyvy ? u : y, q);
}

// Work item idx -> frame f, chroma row c (frame rows ROWS c .. ROWS c + ROWS - 1), first pixel x0 of the group.
__device__ __forceinline__ void yuv_item(long long idx, int groups, int chroma_rows, int& f, int& c, int& x0) {
  const long long rest = idx / groups;
  x0 = static_cast<int>(idx - rest * groups) * kYuvGroup;
  c = static_cast<int>(rest % chroma_rows);
  f = static_cast<int>(rest / chroma_rows);
}

// Register note.  ptxas allocates these kernels' registers differently for small changes in how the row addresses are formed.  Four
// choices keep every instantiation at or below the registers of the per-format bodies the templates replaced:
//   - y_step is the last field of YuvPlanes;
//   - each path of the decode sets its rows' start addresses once, before it uses them;
//   - the encode sets them once for both paths;
//   - store_planar writes its rows out rather than looping over them.
// The straightforward forms give the 8-bit 4:2:0 pc decodes 80 registers instead of 64 (3 CTAs of 256 per SM instead of 4), and the
// 10-bit 4:2:0 encodes up to 59 instead of 48 (4 CTAs instead of 5).
template <class T, int ROWS, class Map>
__global__ void __launch_bounds__(256) yuv_to_bgr_kernel(const YuvPlanes<T> p, int n, int h, int w, T* __restrict__ bgr) {
  using S = Samples<T>;
  constexpr bool kPackable = sizeof(T) == 1 && ROWS == 1;
  const Map m{};
  const int groups = (w + kYuvGroup - 1) / kYuvGroup, chroma_rows = h / ROWS, y_step = kPackable ? p.y_step : 1;
  const long long total = static_cast<long long>(n) * chroma_rows * groups;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    int f, c, x0;
    yuv_item(idx, groups, chroma_rows, f, c, x0);
    const long long fo = f * p.frame_stride;
    const T* y = p.y + fo + static_cast<long long>(ROWS * c) * p.y_pitch + x0 * y_step;
    const long long co = fo + static_cast<long long>(c) * p.c_pitch + (x0 >> 1) * p.c_step;
    const T* u = p.u + co;
    const T* v = p.v + co;
    T* o = bgr + ((static_cast<long long>(f) * h + ROWS * c) * w + x0) * 3;
    if (x0 + kYuvGroup <= w) {
      const T* yr[ROWS];
      T* orow[ROWS];
#pragma unroll
      for (int r = 0; r < ROWS; ++r) {
        yr[r] = y + r * p.y_pitch;
        orow[r] = o + static_cast<long long>(r) * w * 3;
      }
      uint32_t yw[ROWS][S::kRow], uw[S::kChroma], vw[S::kChroma];
      if constexpr (kPackable) {
        if (y_step == 2) load_packed(y, u, yw[0], uw, vw);
        else load_planar(yr, u, v, p.c_step, yw, uw, vw);
      } else {
        load_planar(yr, u, v, p.c_step, yw, uw, vw);
      }
      typename Map::Chroma ch[kYuvGroup / 2];
#pragma unroll
      for (int k = 0; k < kYuvGroup / 2; ++k) ch[k] = m.chroma(S::value(S::at(uw, k), p.msb), S::value(S::at(vw, k), p.msb));
#pragma unroll
      for (int r = 0; r < ROWS; ++r) {             // one row at a time: the row's 24 or 48 output bytes stay in 6 or 12 registers
        uint32_t out[3 * S::kRow] = {};
#pragma unroll
        for (int j = 0; j < kYuvGroup; ++j) {
          int B, G, R;
          m.pixel(ch[j >> 1], S::value(S::at(yw[r], j), p.msb), B, G, R);
          S::put(out, 3 * j, B); S::put(out, 3 * j + 1, G); S::put(out, 3 * j + 2, R);
        }
        store_bytes<12 * S::kRow>(as_bytes(orow[r]), out);
      }
    } else {
      const T* yr[ROWS];
      T* orow[ROWS];
#pragma unroll
      for (int r = 0; r < ROWS; ++r) {
        yr[r] = y + r * p.y_pitch;
        orow[r] = o + static_cast<long long>(r) * w * 3;
      }
      for (int j = 0; x0 + j < w; j += 2) {
        const typename Map::Chroma ch = m.chroma(S::value(u[(j >> 1) * p.c_step], p.msb), S::value(v[(j >> 1) * p.c_step], p.msb));
#pragma unroll
        for (int d = 0; d < 2; ++d) {
#pragma unroll
          for (int r = 0; r < ROWS; ++r) {
            int B, G, R;
            m.pixel(ch, S::value(yr[r][(j + d) * y_step], p.msb), B, G, R);
            T* q = orow[r] + 3 * (j + d);
            q[0] = B; q[1] = G; q[2] = R;
          }
        }
      }
    }
  }
}

template <class T, int ROWS, class Map>
__global__ void __launch_bounds__(256) bgr_to_yuv_kernel(const T* __restrict__ bgr, int n, int h, int w, const YuvPlanes<T> p) {
  using S = Samples<T>;
  constexpr bool kPackable = sizeof(T) == 1 && ROWS == 1;
  const Map m{};
  const int groups = (w + kYuvGroup - 1) / kYuvGroup, chroma_rows = h / ROWS, y_step = kPackable ? p.y_step : 1;
  const long long total = static_cast<long long>(n) * chroma_rows * groups;
  const int sh = S::shift(p.msb);
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    int f, c, x0;
    yuv_item(idx, groups, chroma_rows, f, c, x0);
    const long long fo = f * p.frame_stride;
    T* y = p.y + fo + static_cast<long long>(ROWS * c) * p.y_pitch + x0 * y_step;
    const long long co = fo + static_cast<long long>(c) * p.c_pitch + (x0 >> 1) * p.c_step;
    T* u = p.u + co;
    T* v = p.v + co;
    const T* in = bgr + ((static_cast<long long>(f) * h + ROWS * c) * w + x0) * 3;
    T* yr[ROWS];                                   // where the thread's rows start, for both paths
    const T* irow[ROWS];
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
      yr[r] = y + r * p.y_pitch;
      irow[r] = in + static_cast<long long>(r) * w * 3;
    }
    if (x0 + kYuvGroup <= w) {
      uint32_t iw[ROWS][3 * S::kRow];
#pragma unroll
      for (int r = 0; r < ROWS; ++r) load_bytes<12 * S::kRow>(as_bytes(irow[r]), iw[r]);
      uint32_t yw[ROWS][S::kRow] = {}, uw[S::kChroma] = {}, vw[S::kChroma] = {};
#pragma unroll
      for (int j = 0; j < kYuvGroup; ++j) {
#pragma unroll
        for (int r = 0; r < ROWS; ++r) {
          const int B = S::at(iw[r], 3 * j), G = S::at(iw[r], 3 * j + 1), R = S::at(iw[r], 3 * j + 2);
          S::put(yw[r], j, m.y(R, G, B) << sh);
          if (r == 0 && (j & 1) == 0) {            // the left pixel of its pair, in the first row
            S::put(uw, j >> 1, m.u(R, G, B) << sh);
            S::put(vw, j >> 1, m.v(R, G, B) << sh);
          }
        }
      }
      if constexpr (kPackable) {
        if (y_step == 2) store_packed(y, u, yw[0], uw, vw);
        else store_planar(yr, u, v, p.c_step, yw, uw, vw);
      } else {
        store_planar(yr, u, v, p.c_step, yw, uw, vw);
      }
    } else {
      for (int j = 0; x0 + j < w; j += 2) {
        const T* a = in + 3 * j;
        u[(j >> 1) * p.c_step] = static_cast<T>(m.u(a[2], a[1], a[0]) << sh);
        v[(j >> 1) * p.c_step] = static_cast<T>(m.v(a[2], a[1], a[0]) << sh);
#pragma unroll
        for (int d = 0; d < 2; ++d) {
#pragma unroll
          for (int r = 0; r < ROWS; ++r) {
            const T* q = irow[r] + 3 * (j + d);
            yr[r][(j + d) * y_step] = static_cast<T>(m.y(q[2], q[1], q[0]) << sh);
          }
        }
      }
    }
  }
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

// ------------------------------------------------------------------------------------------------ host side
template <class T>
using DecodeKernel = void (*)(const YuvPlanes<T>, int, int, int, T*);
template <class T>
using EncodeKernel = void (*)(const T*, int, int, int, const YuvPlanes<T>);

// The kernels of each (colorspace, range) for one sample type and subsampling: [BT601][TV] is the cv2-exact map, the others are the
// pair's H.273 maps.
#define SAVSR_CS_TABLE(kernel, T, ROWS)                                                                                    \
  {{kernel<T, ROWS, Cv2Map<T>>, kernel<T, ROWS, CsMap<T, 0, 1>>}, {kernel<T, ROWS, CsMap<T, 1, 0>>, kernel<T, ROWS, CsMap<T, 1, 1>>}, \
   {kernel<T, ROWS, CsMap<T, 2, 0>>, kernel<T, ROWS, CsMap<T, 2, 1>>}}
template <class T, int ROWS>
static const DecodeKernel<T> kDecode[3][2] = SAVSR_CS_TABLE(yuv_to_bgr_kernel, T, ROWS);
template <class T, int ROWS>
static const EncodeKernel<T> kEncode[3][2] = SAVSR_CS_TABLE(bgr_to_yuv_kernel, T, ROWS);
#undef SAVSR_CS_TABLE

// The kernel of (colorspace, range), or an error naming a value not in enum savsr_colorspace / savsr_color_range.
template <class F>
static int cs_kernel(const char* fn, int colorspace, int range, const F (&table)[3][2], F* k) {
  SAVSR_REQUIRE(colorspace >= SAVSR_COLORSPACE_BT601 && colorspace <= SAVSR_COLORSPACE_BT2020NC,
                "%s: unknown colorspace %d (0 BT601, 1 BT709, 2 BT2020NC)", fn, colorspace);
  SAVSR_REQUIRE(range == SAVSR_RANGE_TV || range == SAVSR_RANGE_PC, "%s: unknown color range %d (0 TV, 1 PC)", fn, range);
  *k = table[colorspace][range];
  return 0;
}

// The checks of the plane description and frame size, in the order the entry points make them before any launch.
template <class T, int ROWS>
static int check_yuv(const char* fn, const YuvPlanes<T>& p, int n, int h, int w) {
  constexpr bool deep = sizeof(T) == 2;
  const char* planar = ROWS == 2 ? (deep ? "yuv420p10le" : "yuv420p") : (deep ? "yuv422p10le" : "yuv422p");
  const char* interleaved = ROWS == 2 ? (deep ? "p010" : "nv12") : (deep ? "p210" : "nv16");
  const char* unit = deep ? "elements" : "bytes";
  SAVSR_REQUIRE(n >= 0 && h > 0 && w > 0, "%s: bad shape n=%d h=%d w=%d", fn, n, h, w);
  if (ROWS == 2) {                                 // the 4:2:0 entry points take no y_step: it is 1
    SAVSR_REQUIRE(h % 2 == 0 && w % 2 == 0, "%s: YUV 4:2:0 needs an even frame size, got %dx%d", fn, h, w);
    SAVSR_REQUIRE(p.c_step == 1 || p.c_step == 2, "%s: c_step must be 1 (%s) or 2 (%s), got %d", fn, planar, interleaved, p.c_step);
  } else {
    SAVSR_REQUIRE(w % 2 == 0, "%s: YUV 4:2:2 needs an even width, got %dx%d", fn, h, w);
    SAVSR_REQUIRE((p.y_step == 1 && (p.c_step == 1 || p.c_step == 2)) || (!deep && p.y_step == 2 && p.c_step == 4),
                  "%s: (y_step, c_step) must be (1, 1) (%s), (1, 2) (%s)%s, got (%d, %d)", fn, planar, interleaved,
                  deep ? "" : " or (2, 4) (yuyv422, uyvy422)", p.y_step, p.c_step);
  }
  SAVSR_REQUIRE(p.y_pitch >= p.y_step * w, "%s: y_pitch %d < row of %d %s", fn, p.y_pitch, p.y_step * w, unit);
  SAVSR_REQUIRE(p.c_pitch >= p.c_step * (w / 2), "%s: c_pitch %d < chroma row of %d %s", fn, p.c_pitch, p.c_step * (w / 2), unit);
  // Only 4:2:2 requires v = u + 1 of interleaved chroma; the 4:2:0 entry points have always taken v as given.
  SAVSR_REQUIRE(ROWS == 2 || p.c_step != 2 || p.v == p.u + 1, "%s: interleaved chroma (c_step 2) needs v = u + 1", fn);
  SAVSR_REQUIRE(p.y_step != 2 || (p.c_pitch == p.y_pitch && ((p.u == p.y + 1 && p.v == p.y + 3) || (p.u == p.y - 1 && p.v == p.y + 1))),
                "%s: packed 4:2:2 needs c_pitch = y_pitch and yuyv422 (u = y + 1, v = y + 3) or uyvy422 (u = y - 1, v = y + 1)", fn);
  SAVSR_REQUIRE(p.frame_stride >= 0, "%s: negative frame_stride %lld", fn, p.frame_stride);
  if (deep) SAVSR_REQUIRE(p.msb == 0 || p.msb == 1, "%s: msb must be 0 (%s) or 1 (%s), got %d", fn, planar, interleaved, p.msb);
  return 0;
}

template <class T>
static YuvPlanes<T> planes(const T* y, int y_pitch, int y_step, const T* u, const T* v, int c_pitch, int c_step, long long frame_stride,
                           int msb) {
  return {const_cast<T*>(y), const_cast<T*>(u), const_cast<T*>(v), y_pitch, c_pitch, c_step, frame_stride, msb, y_step};
}

static unsigned grid_for(const savsr_ctx* ctx, long long items) {
  const long long b = (items + 255) / 256, cap = 16LL * ctx->sm_count;
  return static_cast<unsigned>(b < cap ? b : cap);
}

// The two conversions: the colour pair's kernel, the null and layout checks, then one launch over n * (h / ROWS) * groups items.
template <class T, int ROWS>
static int yuv_to_bgr(const char* fn, savsr_ctx* ctx, const YuvPlanes<T>& p, int n, int h, int w, T* bgr, int colorspace, int range,
                      savsr_stream st) {
  DecodeKernel<T> k;
  if (cs_kernel(fn, colorspace, range, kDecode<T, ROWS>, &k)) return 1;
  SAVSR_REQUIRE(ctx && p.y && p.u && p.v && bgr, "%s: null pointer", fn);
  if (check_yuv<T, ROWS>(fn, p, n, h, w)) return 1;
  if (n == 0) return 0;
  DeviceGuard guard(ctx->device);
  const long long items = static_cast<long long>(n) * (h / ROWS) * ((w + kYuvGroup - 1) / kYuvGroup);
  k<<<grid_for(ctx, items), 256, 0, static_cast<cudaStream_t>(st)>>>(p, n, h, w, bgr);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

template <class T, int ROWS>
static int bgr_to_yuv(const char* fn, savsr_ctx* ctx, const T* bgr, int n, int h, int w, const YuvPlanes<T>& p, int colorspace, int range,
                      savsr_stream st) {
  EncodeKernel<T> k;
  if (cs_kernel(fn, colorspace, range, kEncode<T, ROWS>, &k)) return 1;
  SAVSR_REQUIRE(ctx && bgr && p.y && p.u && p.v, "%s: null pointer", fn);
  if (check_yuv<T, ROWS>(fn, p, n, h, w)) return 1;
  if (n == 0) return 0;
  DeviceGuard guard(ctx->device);
  const long long items = static_cast<long long>(n) * (h / ROWS) * ((w + kYuvGroup - 1) / kYuvGroup);
  k<<<grid_for(ctx, items), 256, 0, static_cast<cudaStream_t>(st)>>>(bgr, n, h, w, p);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace savsr

using namespace savsr;

// The plain 4:2:0 entry points convert the default pair, (BT601, TV); the _cs ones check the pair they are given first.
extern "C" int savsr_yuv420_to_bgr(savsr_ctx* ctx, const uint8_t* y, int y_pitch, const uint8_t* u, const uint8_t* v, int c_pitch,
                                   int c_step, int64_t frame_stride, int n, int h, int w, uint8_t* bgr, savsr_stream st) {
  return yuv_to_bgr<uint8_t, 2>("savsr_yuv420_to_bgr", ctx, planes(y, y_pitch, 1, u, v, c_pitch, c_step, frame_stride, 0), n, h, w, bgr,
                                SAVSR_COLORSPACE_BT601, SAVSR_RANGE_TV, st);
}

extern "C" int savsr_yuv420_to_bgr_cs(savsr_ctx* ctx, const uint8_t* y, int y_pitch, const uint8_t* u, const uint8_t* v, int c_pitch,
                                      int c_step, int64_t frame_stride, int n, int h, int w, uint8_t* bgr, int colorspace, int range,
                                      savsr_stream st) {
  return yuv_to_bgr<uint8_t, 2>("savsr_yuv420_to_bgr_cs", ctx, planes(y, y_pitch, 1, u, v, c_pitch, c_step, frame_stride, 0), n, h, w, bgr,
                                colorspace, range, st);
}

extern "C" int savsr_bgr_to_yuv420(savsr_ctx* ctx, const uint8_t* bgr, int n, int h, int w, uint8_t* y, int y_pitch, uint8_t* u, uint8_t* v,
                                   int c_pitch, int c_step, int64_t frame_stride, savsr_stream st) {
  return bgr_to_yuv<uint8_t, 2>("savsr_bgr_to_yuv420", ctx, bgr, n, h, w, planes<uint8_t>(y, y_pitch, 1, u, v, c_pitch, c_step, frame_stride, 0),
                                SAVSR_COLORSPACE_BT601, SAVSR_RANGE_TV, st);
}

extern "C" int savsr_bgr_to_yuv420_cs(savsr_ctx* ctx, const uint8_t* bgr, int n, int h, int w, uint8_t* y, int y_pitch, uint8_t* u,
                                      uint8_t* v, int c_pitch, int c_step, int64_t frame_stride, int colorspace, int range, savsr_stream st) {
  return bgr_to_yuv<uint8_t, 2>("savsr_bgr_to_yuv420_cs", ctx, bgr, n, h, w,
                                planes<uint8_t>(y, y_pitch, 1, u, v, c_pitch, c_step, frame_stride, 0), colorspace, range, st);
}

extern "C" int savsr_yuv420_10_to_bgr48(savsr_ctx* ctx, const uint16_t* y, int y_pitch, const uint16_t* u, const uint16_t* v, int c_pitch,
                                        int c_step, int64_t frame_stride, int msb, int n, int h, int w, uint16_t* bgr, savsr_stream st) {
  return yuv_to_bgr<uint16_t, 2>("savsr_yuv420_10_to_bgr48", ctx, planes(y, y_pitch, 1, u, v, c_pitch, c_step, frame_stride, msb), n, h, w,
                                 bgr, SAVSR_COLORSPACE_BT601, SAVSR_RANGE_TV, st);
}

extern "C" int savsr_yuv420_10_to_bgr48_cs(savsr_ctx* ctx, const uint16_t* y, int y_pitch, const uint16_t* u, const uint16_t* v,
                                           int c_pitch, int c_step, int64_t frame_stride, int msb, int n, int h, int w, uint16_t* bgr,
                                           int colorspace, int range, savsr_stream st) {
  return yuv_to_bgr<uint16_t, 2>("savsr_yuv420_10_to_bgr48_cs", ctx, planes(y, y_pitch, 1, u, v, c_pitch, c_step, frame_stride, msb), n, h,
                                 w, bgr, colorspace, range, st);
}

extern "C" int savsr_bgr48_to_yuv420_10(savsr_ctx* ctx, const uint16_t* bgr, int n, int h, int w, uint16_t* y, int y_pitch, uint16_t* u,
                                        uint16_t* v, int c_pitch, int c_step, int64_t frame_stride, int msb, savsr_stream st) {
  return bgr_to_yuv<uint16_t, 2>("savsr_bgr48_to_yuv420_10", ctx, bgr, n, h, w,
                                 planes<uint16_t>(y, y_pitch, 1, u, v, c_pitch, c_step, frame_stride, msb), SAVSR_COLORSPACE_BT601,
                                 SAVSR_RANGE_TV, st);
}

extern "C" int savsr_bgr48_to_yuv420_10_cs(savsr_ctx* ctx, const uint16_t* bgr, int n, int h, int w, uint16_t* y, int y_pitch, uint16_t* u,
                                           uint16_t* v, int c_pitch, int c_step, int64_t frame_stride, int msb, int colorspace, int range,
                                           savsr_stream st) {
  return bgr_to_yuv<uint16_t, 2>("savsr_bgr48_to_yuv420_10_cs", ctx, bgr, n, h, w,
                                 planes<uint16_t>(y, y_pitch, 1, u, v, c_pitch, c_step, frame_stride, msb), colorspace, range, st);
}

extern "C" int savsr_yuv422_to_bgr_cs(savsr_ctx* ctx, const uint8_t* y, int y_pitch, int y_step, const uint8_t* u, const uint8_t* v,
                                      int c_pitch, int c_step, int64_t frame_stride, int n, int h, int w, uint8_t* bgr, int colorspace,
                                      int range, savsr_stream st) {
  return yuv_to_bgr<uint8_t, 1>("savsr_yuv422_to_bgr_cs", ctx, planes(y, y_pitch, y_step, u, v, c_pitch, c_step, frame_stride, 0), n, h, w,
                                bgr, colorspace, range, st);
}

extern "C" int savsr_bgr_to_yuv422_cs(savsr_ctx* ctx, const uint8_t* bgr, int n, int h, int w, uint8_t* y, int y_pitch, int y_step,
                                      uint8_t* u, uint8_t* v, int c_pitch, int c_step, int64_t frame_stride, int colorspace, int range,
                                      savsr_stream st) {
  return bgr_to_yuv<uint8_t, 1>("savsr_bgr_to_yuv422_cs", ctx, bgr, n, h, w,
                                planes<uint8_t>(y, y_pitch, y_step, u, v, c_pitch, c_step, frame_stride, 0), colorspace, range, st);
}

extern "C" int savsr_yuv422_10_to_bgr48_cs(savsr_ctx* ctx, const uint16_t* y, int y_pitch, int y_step, const uint16_t* u, const uint16_t* v,
                                           int c_pitch, int c_step, int64_t frame_stride, int msb, int n, int h, int w, uint16_t* bgr,
                                           int colorspace, int range, savsr_stream st) {
  return yuv_to_bgr<uint16_t, 1>("savsr_yuv422_10_to_bgr48_cs", ctx, planes(y, y_pitch, y_step, u, v, c_pitch, c_step, frame_stride, msb),
                                 n, h, w, bgr, colorspace, range, st);
}

extern "C" int savsr_bgr48_to_yuv422_10_cs(savsr_ctx* ctx, const uint16_t* bgr, int n, int h, int w, uint16_t* y, int y_pitch, int y_step,
                                           uint16_t* u, uint16_t* v, int c_pitch, int c_step, int64_t frame_stride, int msb,
                                           int colorspace, int range, savsr_stream st) {
  return bgr_to_yuv<uint16_t, 1>("savsr_bgr48_to_yuv422_10_cs", ctx, bgr, n, h, w,
                                 planes<uint16_t>(y, y_pitch, y_step, u, v, c_pitch, c_step, frame_stride, msb), colorspace, range, st);
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
