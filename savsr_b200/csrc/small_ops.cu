// CUDA-core kernels around the tensor-core convolutions: first-layer convs on the fp32 input window,
// the OSA-Conv prologue (pool -> scale_routing MLP -> ScaleAttention -> per-sample kernel assembly),
// RCAB channel attention, and the OSAdapt mask tail.  All HBM/L2-bound or latency-bound by nature;
// they use coalesced 128-bit accesses and keep weights in shared memory.
#include <type_traits>

#include "common.cuh"

namespace savsr {

// ------------------------------------------------------------------------------------------------ first layer: frame packing
// The input window -> one bf16 arena slot whose channels 0..3t-1 are the frames' RGB planes (channel 3f + c), the rest zero,
// reflect-padded to the even arena size (savsr_arch.py:670-690).  With this slot the first-layer convs (conv_c / conv_sup,
// savsr_arch.py:456-457) run on the tensor-core kernel with zero-expanded weights.  T = float: fp32 NCHW window [B][t][3][h][w] RGB;
// T = uint8_t: the decoded 8-bit window [B][t][h][w][3] BGR, converted exactly as the reference's img.astype(np.float32) / 255.;
// T = const uint8_t*: a frame table (x[n * t + f] -> frame f of sample n, [h][w][3] BGR), read through the same conversion;
// T = const uint16_t*: a frame table of bgr48 frames, read through u16_to_unit (v / 65535, correctly rounded).
template <class T>
__global__ void __launch_bounds__(256) pack_frames_kernel(const T* __restrict__ x, __nv_bfloat16* __restrict__ dst, int batch,
                                                          int t, int h, int w, int hp, int wp, int fmt) {
  const long npix = static_cast<long>(hp) * wp;
  const long total = static_cast<long>(batch) * npix * 8;
  for (long id = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; id < total; id += static_cast<long>(gridDim.x) * blockDim.x) {
    const int chunk = id & 7;
    const long pn = id >> 3;
    const long pix = pn % npix;
    const int n = pn / npix;
    const int py = pix / wp, px = pix % wp;
    const int ry = py < h ? py : 2 * h - 2 - py, rx = px < w ? px : 2 * w - 2 - px;
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int ch = chunk * 8 + e;
      if constexpr (std::is_pointer<T>::value) {
        const int f = ch / 3, c = ch - 3 * f;
        v[e] = ch < 3 * t ? to_unit(__ldg(frame_at(x, static_cast<long>(n) * t + f) + (static_cast<long>(ry) * w + rx) * 3 + 2 - c)) : 0.f;
      } else if constexpr (sizeof(T) == 1) {
        const int f = ch / 3, c = ch - 3 * f;
        v[e] = ch < 3 * t ? u8_to_unit(__ldg(x + ((static_cast<long>(n) * t + f) * h + ry) * w * 3 + rx * 3 + 2 - c)) : 0.f;
      } else {
        v[e] = ch < 3 * t ? __ldg(x + ((static_cast<long>(n) * t * 3 + ch) * h + ry) * w + rx) : 0.f;
      }
    }
    uint4 o;
    o.x = pack_h2(v[0], v[1], fmt); o.y = pack_h2(v[2], v[3], fmt); o.z = pack_h2(v[4], v[5], fmt); o.w = pack_h2(v[6], v[7], fmt);
    *reinterpret_cast<uint4*>(dst + (static_cast<long>(n) * npix + pix) * kC + chunk * 8) = o;
  }
}

// ------------------------------------------------------------------------------------------------ OSA prologue
constexpr int kMaxOsa = 4;
struct OsaLaunch {
  savsr_osa_params c[kMaxOsa];
  int nconvs, batch, npart, npix;
  float inv_h, inv_w;
  int fmt;
};
__host__ __device__ inline int osa_scratch_stride(int ci) { return 5 * ci + 192; }
__host__ __device__ inline int osa_off_h1(int ci) { return ci + 8; }
__host__ __device__ inline int osa_off_v2(int ci) { return 3 * ci + 8; }
__host__ __device__ inline int osa_off_att(int ci) { return 4 * ci + 8; }

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

// vin = [1/s_h, 1/s_w, mean(x)] (savsr_arch.py:143-146), mean from the producers' partial sums.
// grid (nsrc_max, batch, nconvs), 1024 threads = 16 partial ranges x 64 channels.
constexpr int kOsaThreads = 1024;
__global__ void __launch_bounds__(kOsaThreads) osa_pool_kernel(const __grid_constant__ OsaLaunch L) {
  pdl_wait();
  pdl_trigger();
  const savsr_osa_params& c = L.c[blockIdx.z];
  const int s = blockIdx.x, n = blockIdx.y;
  if (s * 64 >= c.ci) return;
  __shared__ float red[16][64];
  const int ch = threadIdx.x & 63, part = threadIdx.x >> 6;
  const float* src = c.pool[s] + static_cast<long>(n) * L.npart * kC;
  float a0 = 0.f, a1 = 0.f;
  int q = part;
  for (; q + 16 < L.npart; q += 32) { a0 += src[q * kC + ch]; a1 += src[(q + 16) * kC + ch]; }
  if (q < L.npart) a0 += src[q * kC + ch];
  red[part][ch] = a0 + a1;
  __syncthreads();
  float* vin = c.scratch + static_cast<long>(n) * osa_scratch_stride(c.ci);
  if (part == 0) {
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) sum += red[k][ch];
    vin[2 + s * 64 + ch] = sum / static_cast<float>(L.npix);
  }
  if (s == 0 && threadIdx.x == 0) { vin[0] = L.inv_h; vin[1] = L.inv_w; }
}

// One Linear + ReLU layer of scale_routing (savsr_arch.py:123-128).  layer 0: [2ci][ci+2], layer 1: [ci][2ci].
// grid (row blocks, nconvs), 256 threads = 8 warps, one output row per warp.  The inputs of ALL samples are staged in
// shared memory and the row's weights sit in registers, so each weight is fetched once and every sample costs one
// shared-memory dot product + shuffle reduction.
__global__ void __launch_bounds__(256) osa_linear_kernel(const __grid_constant__ OsaLaunch L, int layer) {
  pdl_wait();
  pdl_trigger();
  extern __shared__ float s_in[];   // [batch][len]
  const savsr_osa_params& c = L.c[blockIdx.y];
  const int rows = layer == 0 ? 2 * c.ci : c.ci;
  const int len = layer == 0 ? c.ci + 2 : 2 * c.ci;
  const int in_off = layer == 0 ? 0 : osa_off_h1(c.ci);
  const int out_off = layer == 0 ? osa_off_h1(c.ci) : osa_off_v2(c.ci);
  const float* W = layer == 0 ? c.r0_w : c.r2_w;
  const float* B = layer == 0 ? c.r0_b : c.r2_b;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (blockIdx.x * 8 >= rows) return;
  const int stride = osa_scratch_stride(c.ci);
  // samples are split over blockIdx.z: 24-48 row blocks alone leave most SMs idle and each warp walking all samples
  const int per = (L.batch + gridDim.z - 1) / gridDim.z;
  const int n0 = blockIdx.z * per, n1 = min(L.batch, n0 + per);
  if (n0 >= n1) return;
  for (int i = threadIdx.x; i < (n1 - n0) * len; i += blockDim.x) {
    const int n = i / len, k = i - n * len;
    s_in[i] = c.scratch[static_cast<long>(n0 + n) * stride + in_off + k];
  }
  __syncthreads();
  const int row = blockIdx.x * 8 + warp;
  if (row >= rows) return;
  const float* wr = W + static_cast<long>(row) * len;
  float w[20];   // ceil(640 / 32)
#pragma unroll
  for (int j = 0; j < 20; ++j) w[j] = lane + 32 * j < len ? __ldg(wr + lane + 32 * j) : 0.f;
  const float bias = B[row];
  for (int n = n0; n < n1; ++n) {
    const float* in = s_in + (n - n0) * len;
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < 20; ++j) if (lane + 32 * j < len) acc += w[j] * in[lane + 32 * j];
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (lane == 0) c.scratch[static_cast<long>(n) * stride + out_off + row] = fmaxf(acc + bias, 0.f);
  }
}

// ScaleAttention + kernel assembly in one launch.  W'[o,i,u,v] = fa[o] ca[i] sa[u,v] sum_k ka[k] bank[k,o,i,u,v]  -> packed
// 16-bit K-blocks (n_tile 64, SAVSR_ROWS_QUAD).  grid (ceil(co*ci/256), nconvs, sample splits), thread = (o, i) with its 72
// bank values in registers across the samples of the split.  Every block first recomputes the attention vectors of its
// samples in shared memory (z = ReLU(BN(fc v)), sigmoid heads ca / fa / sa, softmax head ka: ~5 kMAC per sample, far
// cheaper than a separate launch); block x = 0 also writes them to the scratch area (tests read them there).
constexpr int kAsmMaxSamples = 8;
__global__ void __launch_bounds__(256) osa_assemble_kernel(const __grid_constant__ OsaLaunch L) {
  const savsr_osa_params& c = L.c[blockIdx.y];
  __shared__ float z_s[kAsmMaxSamples][32];
  __shared__ float att_s[kAsmMaxSamples][64 * SAVSR_MAX_SRC + 64 + 9 + 8];
  const int per = (L.batch + gridDim.z - 1) / gridDim.z;       // <= kAsmMaxSamples (checked by the launcher)
  const int n0 = blockIdx.z * per, n1 = min(L.batch, n0 + per);
  if (n0 >= n1 || blockIdx.x * blockDim.x >= c.co * c.ci) return;
  const int ns = n1 - n0;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int stride = osa_scratch_stride(c.ci);
  const int nout = c.ci + c.co + 9 + 8;
  // z[n][a] (savsr_arch.py:91-93): one warp per attention channel, its fc row held in registers across the samples
  for (int a = warp; a < c.att; a += 8) {
    float wr[10];   // ceil(320 / 32)
#pragma unroll
    for (int j = 0; j < 10; ++j) wr[j] = lane + 32 * j < c.ci ? __ldg(c.fc_w + a * c.ci + lane + 32 * j) : 0.f;
    const float bs = c.bn_scale[a], bh = c.bn_shift[a];
    for (int n = 0; n < ns; ++n) {
      const float* v2 = c.scratch + static_cast<long>(n0 + n) * stride + osa_off_v2(c.ci);
      float acc = 0.f;
#pragma unroll
      for (int j = 0; j < 10; ++j) if (lane + 32 * j < c.ci) acc += wr[j] * v2[lane + 32 * j];
#pragma unroll
      for (int off = 16; off >= 1; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
      if (lane == 0) z_s[n][a] = fmaxf(acc * bs + bh, 0.f);
    }
  }
  __syncthreads();
  // heads (94-96): sigmoid for channel / filter / spatial, logits for the kernel head; one output per thread, its weight row
  // (att <= 32 floats) loaded once and applied to every sample of the split
  for (int j = threadIdx.x; j < nout; j += blockDim.x) {
    const float* w;
    float b;
    if (j < c.ci) { w = c.ch_w + j * c.att; b = c.ch_b[j]; }
    else if (j < c.ci + c.co) { w = c.fl_w + (j - c.ci) * c.att; b = c.fl_b[j - c.ci]; }
    else if (j < c.ci + c.co + 9) { w = c.sp_w + (j - c.ci - c.co) * c.att; b = c.sp_b[j - c.ci - c.co]; }
    else { w = c.kn_w + (j - c.ci - c.co - 9) * c.att; b = c.kn_b[j - c.ci - c.co - 9]; }
    float wv[32];
#pragma unroll
    for (int a = 0; a < 32; ++a) wv[a] = a < c.att ? __ldg(w + a) : 0.f;
    const bool sig = j < c.ci + c.co + 9;
    for (int n = 0; n < ns; ++n) {
      float acc = b;
#pragma unroll
      for (int a = 0; a < 32; ++a) if (a < c.att) acc += wv[a] * z_s[n][a];
      att_s[n][j] = sig ? sigmoidf_(acc) : acc;
    }
  }
  __syncthreads();
  if (threadIdx.x < ns) {   // softmax over the 8 kernel logits (temperature 1)
    float* ka = att_s[threadIdx.x] + c.ci + c.co + 9;
    float mx = ka[0];
    for (int k = 1; k < 8; ++k) mx = fmaxf(mx, ka[k]);
    float e[8], sum = 0.f;
    for (int k = 0; k < 8; ++k) { e[k] = expf(ka[k] - mx); sum += e[k]; }
    for (int k = 0; k < 8; ++k) ka[k] = e[k] / sum;
  }
  __syncthreads();
  if (blockIdx.x == 0) {
    for (int r = threadIdx.x; r < ns * nout; r += blockDim.x) {
      const int n = r / nout, j = r - n * nout;
      c.scratch[static_cast<long>(n0 + n) * stride + osa_off_att(c.ci) + j] = att_s[n][j];
    }
  }
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= c.co * c.ci) return;
  const int i = idx % c.ci, o = idx / c.ci;
  float bk[8][9];
  const long per_k = static_cast<long>(c.co) * c.ci * 9;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float* src = c.bank + k * per_k + (static_cast<long>(o) * c.ci + i) * 9;
#pragma unroll
    for (int t = 0; t < 9; ++t) bk[k][t] = __ldg(src + t);
  }
  const int s = i >> 6, kk = i & 63;
  const long sample_elems = static_cast<long>(c.co) * c.ci * 9;
  const int row = quad_row(o);   // SAVSR_ROWS_QUAD: the packed row that holds output channel o (the map is an involution)
  const int inner = row * 64 + ((((kk >> 3) ^ (row & 7)) << 3) | (kk & 7));
  for (int n = 0; n < ns; ++n) {
    const float* att = att_s[n];
    const float ca = att[i], fa = att[c.ci + o];
    const float* sa = att + c.ci + c.co;
    const float* ka = sa + 9;
    uint16_t* dst = static_cast<uint16_t*>(c.packed) + (n0 + n) * sample_elems;
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      float acc = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) acc += ka[k] * bk[k][t];
      dst[static_cast<long>(s * 9 + t) * 4096 + inner] = float_to_h(acc * sa[t] * ca * fa, L.fmt);
    }
  }
}

// ------------------------------------------------------------------------------------------------ RCAB channel attention
struct CaParams {
  const __nv_bfloat16* t;
  const __nv_bfloat16* x;
  __nv_bfloat16* dst;
  const float* pool;
  const float *w1, *b1, *w2, *b2;
  float* y;      // [batch][64] channel scales (scratch)
  int npart;
  int fmt;
  long npix;
};
// y = sigmoid(W2 relu(W1 mean(t) + b1) + b2) per sample (savsr_arch.py:514-519).  grid (batch), 1024 threads.
__global__ void __launch_bounds__(1024) ca_vector_kernel(const CaParams p) {
  pdl_wait();
  pdl_trigger();
  __shared__ float red[16][64];
  __shared__ float mean[64];
  __shared__ float hid[4];
  const int n = blockIdx.x;
  const int ch = threadIdx.x & 63, part = threadIdx.x >> 6;
  const float* src = p.pool + static_cast<long>(n) * p.npart * kC;
  float a0 = 0.f, a1 = 0.f;
  int q = part;
  for (; q + 16 < p.npart; q += 32) { a0 += src[q * kC + ch]; a1 += src[(q + 16) * kC + ch]; }
  if (q < p.npart) a0 += src[q * kC + ch];
  red[part][ch] = a0 + a1;
  __syncthreads();
  if (part == 0) {
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) sum += red[k][ch];
    mean[ch] = sum / static_cast<float>(p.npix);
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    float a = p.b1[threadIdx.x];
    for (int i = 0; i < 64; ++i) a += p.w1[threadIdx.x * 64 + i] * mean[i];
    hid[threadIdx.x] = fmaxf(a, 0.f);
  }
  __syncthreads();
  if (threadIdx.x < 64) {
    float a = p.b2[threadIdx.x];
#pragma unroll
    for (int i = 0; i < 4; ++i) a += p.w2[threadIdx.x * 4 + i] * hid[i];
    p.y[n * 64 + threadIdx.x] = sigmoidf_(a);
  }
}
// dst = x + t * y (savsr_arch.py:524, 547-549), streamed as 16-byte chunks.  grid (blocks, batch), 256 threads.
__global__ void __launch_bounds__(256) ca_scale_residual_kernel(const CaParams p) {
  pdl_wait();
  pdl_trigger();
  __shared__ float ys[64];
  const int n = blockIdx.y;
  if (threadIdx.x < 64) ys[threadIdx.x] = p.y[n * 64 + threadIdx.x];
  __syncthreads();
  const long chunks = p.npix * 8;
  const uint4* tt = reinterpret_cast<const uint4*>(p.t + static_cast<long>(n) * p.npix * kC);
  const uint4* xx = reinterpret_cast<const uint4*>(p.x + static_cast<long>(n) * p.npix * kC);
  uint4* dd = reinterpret_cast<uint4*>(p.dst + static_cast<long>(n) * p.npix * kC);
  for (long id = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; id < chunks;
       id += static_cast<long>(gridDim.x) * blockDim.x) {
    const int c0 = (id & 7) * 8;
    const uint4 a = tt[id], b = xx[id];
    uint4 o;
    o.x = pack_h2(h_lo(b.x, p.fmt) + h_lo(a.x, p.fmt) * ys[c0 + 0], h_hi(b.x, p.fmt) + h_hi(a.x, p.fmt) * ys[c0 + 1], p.fmt);
    o.y = pack_h2(h_lo(b.y, p.fmt) + h_lo(a.y, p.fmt) * ys[c0 + 2], h_hi(b.y, p.fmt) + h_hi(a.y, p.fmt) * ys[c0 + 3], p.fmt);
    o.z = pack_h2(h_lo(b.z, p.fmt) + h_lo(a.z, p.fmt) * ys[c0 + 4], h_hi(b.z, p.fmt) + h_hi(a.z, p.fmt) * ys[c0 + 5], p.fmt);
    o.w = pack_h2(h_lo(b.w, p.fmt) + h_lo(a.w, p.fmt) * ys[c0 + 6], h_hi(b.w, p.fmt) + h_hi(a.w, p.fmt) * ys[c0 + 7], p.fmt);
    dd[id] = o;
  }
}

// OSAdapt mask tail at half resolution (savsr_arch.py:193-205).  Four threads share one half-resolution pixel: thread q
// (= lane & 3) loads input channels 4q..4q+3 of every tap (one float4 per source pixel; nothing is fetched twice), forms
// partial sums of all 16 outputs over its 4 channels, and a shuffle reduce-scatter leaves outputs 4q..4q+3 in thread q.
//   kPool = true : input = AvgPool2d(2) of the full-resolution [B][H][W][16] map, fused into the loads;
//   kProj = true : instead of the 16 ReLU outputs the kernel stores, per pixel, the NINE projections
//                  d[t] = sum_c w_final[t][c] * out[c] of the final 16 -> 1 conv's taps (row stride 12 floats).
// The final conv runs AFTER a bilinear x2 upsample; both are linear, so conv(up(h)) = sum_t up(d_t) shifted by tap t,
// and the full-resolution kernel reads 36 scalars per pixel instead of 36 sixteen-channel vectors.
template <bool kPool, bool kProj>
__global__ void __launch_bounds__(256) mask_conv16_kernel(const float* __restrict__ in, const float* __restrict__ w,
                                                          const float* __restrict__ b, const float* __restrict__ wf,
                                                          float* __restrict__ out, int h2, int w2) {
  // [tap][ci][co] with 16 bytes of padding after every 4 input channels: the four threads of a quad read rows 4q + c,
  // 256 bytes apart without the padding = the same banks, and every LDS.128 would take 16 wavefronts instead of 1
  __shared__ __align__(16) float w_s[9 * 16 * 16 + 36 * 4];
  __shared__ float wf_s[9 * 16];                    // [tap][ci] of the final conv (kProj)
  for (int i = threadIdx.x; i < 9 * 256; i += blockDim.x) {
    const int co = i & 15, ci = (i >> 4) & 15, tap = i >> 8;
    w_s[i + (i >> 6) * 4] = w[(co * 16 + ci) * 9 + tap];
  }
  if (kProj) {
    for (int i = threadIdx.x; i < 144; i += blockDim.x) wf_s[i] = wf[(i & 15) * 9 + (i >> 4)];
  }
  __syncthreads();
  const int n = blockIdx.y;
  const int q = threadIdx.x & 3;
  const long npix2 = static_cast<long>(h2) * w2;
  const long pix = blockIdx.x * static_cast<long>(blockDim.x >> 2) + (threadIdx.x >> 2);
  const bool live = pix < npix2;                    // whole quads are live or not; dead quads still run the shuffles
  const int py = live ? pix / w2 : 0, px = live ? pix % w2 : 0;
  float acc[16];
#pragma unroll
  for (int o = 0; o < 16; ++o) acc[o] = 0.f;
  const int wfull = 2 * w2;
  const float* base = kPool ? in + static_cast<long>(n) * (4 * npix2) * 16 : in + static_cast<long>(n) * npix2 * 16;
#pragma unroll
  for (int tap = 0; tap < 9; ++tap) {
    const int sy = py + tap / 3 - 1, sx = px + tap % 3 - 1;
    if (!live || sy < 0 || sy >= h2 || sx < 0 || sx >= w2) continue;
    float4 a;
    if (kPool) {
      const float4 q0 = *reinterpret_cast<const float4*>(base + (static_cast<long>(2 * sy) * wfull + 2 * sx) * 16 + 4 * q);
      const float4 q1 = *reinterpret_cast<const float4*>(base + (static_cast<long>(2 * sy) * wfull + 2 * sx + 1) * 16 + 4 * q);
      const float4 q2 = *reinterpret_cast<const float4*>(base + (static_cast<long>(2 * sy + 1) * wfull + 2 * sx) * 16 + 4 * q);
      const float4 q3 = *reinterpret_cast<const float4*>(base + (static_cast<long>(2 * sy + 1) * wfull + 2 * sx + 1) * 16 + 4 * q);
      a.x = 0.25f * ((q0.x + q1.x) + (q2.x + q3.x)); a.y = 0.25f * ((q0.y + q1.y) + (q2.y + q3.y));
      a.z = 0.25f * ((q0.z + q1.z) + (q2.z + q3.z)); a.w = 0.25f * ((q0.w + q1.w) + (q2.w + q3.w));
    } else {
      a = *reinterpret_cast<const float4*>(base + (static_cast<long>(sy) * w2 + sx) * 16 + 4 * q);
    }
    const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const float4* wr = reinterpret_cast<const float4*>(w_s + (tap * 16 + 4 * q + c) * 16 + (tap * 4 + q) * 4);
#pragma unroll
      for (int o4 = 0; o4 < 4; ++o4) {
        const float4 wv = wr[o4];
        acc[4 * o4 + 0] += av[c] * wv.x; acc[4 * o4 + 1] += av[c] * wv.y;
        acc[4 * o4 + 2] += av[c] * wv.z; acc[4 * o4 + 3] += av[c] * wv.w;
      }
    }
  }
  // reduce-scatter over the quad: 16 -> 8 (xor 2) -> 4 (xor 1); thread q ends with outputs 4q .. 4q+3
#pragma unroll
  for (int off = 2, cnt = 8; off >= 1; off >>= 1, cnt >>= 1) {
    const bool upper = (q & off) != 0;
#pragma unroll
    for (int i = 0; i < cnt; ++i) {
      const float send = upper ? acc[i] : acc[i + cnt];
      const float keep = upper ? acc[i + cnt] : acc[i];
      acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  float o4v[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) o4v[i] = fmaxf(acc[i] + b[4 * q + i], 0.f);
  if (!kProj) {
    if (live) *reinterpret_cast<float4*>(out + (static_cast<long>(n) * npix2 + pix) * 16 + 4 * q) = make_float4(o4v[0], o4v[1], o4v[2], o4v[3]);
  } else {
    float d[9];
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      float v = 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) v += wf_s[t * 16 + 4 * q + i] * o4v[i];
      v += __shfl_xor_sync(0xffffffffu, v, 1);
      v += __shfl_xor_sync(0xffffffffu, v, 2);
      d[t] = v;
    }
    if (live && q < 3) {
      float* dst = out + (static_cast<long>(n) * npix2 + pix) * 12 + 4 * q;
      *reinterpret_cast<float4*>(dst) = q == 0 ? make_float4(d[0], d[1], d[2], d[3])
                                     : q == 1 ? make_float4(d[4], d[5], d[6], d[7]) : make_float4(d[8], 0.f, 0.f, 0.f);
    }
  }
}

// mask = sigmoid(bias + sum_t bilinear_x2(d_t)(p + tap t)): the bilinear x2 upsample (align_corners = False) of the nine tap
// projections written by mask_conv16_kernel<false, true>, zero outside the full-resolution image (conv padding 1).
__global__ void __launch_bounds__(256) mask_final_kernel(const float* __restrict__ d, const float* __restrict__ b,
                                                         float* __restrict__ mask, int h2, int w2) {
  const int n = blockIdx.y;
  const int H = 2 * h2, W = 2 * w2;
  const long npix = static_cast<long>(H) * W;
  const long pix = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  if (pix >= npix) return;
  const int py = pix / W, px = pix % W;
  const float* base = d + static_cast<long>(n) * h2 * w2 * 12;
  float acc = b[0];
#pragma unroll
  for (int tap = 0; tap < 9; ++tap) {
    const int sy = py + tap / 3 - 1, sx = px + tap % 3 - 1;
    if (sy < 0 || sy >= H || sx < 0 || sx >= W) continue;
    float fy = 0.5f * (static_cast<float>(sy) + 0.5f) - 0.5f;
    float fx = 0.5f * (static_cast<float>(sx) + 0.5f) - 0.5f;
    fy = fy < 0.f ? 0.f : fy;
    fx = fx < 0.f ? 0.f : fx;
    const int y0 = static_cast<int>(fy), x0 = static_cast<int>(fx);
    const int y1 = y0 + (y0 < h2 - 1 ? 1 : 0), x1 = x0 + (x0 < w2 - 1 ? 1 : 0);
    const float ly = fy - y0, lx = fx - x0;
    const float v00 = base[(static_cast<long>(y0) * w2 + x0) * 12 + tap], v01 = base[(static_cast<long>(y0) * w2 + x1) * 12 + tap];
    const float v10 = base[(static_cast<long>(y1) * w2 + x0) * 12 + tap], v11 = base[(static_cast<long>(y1) * w2 + x1) * 12 + tap];
    acc += (1.f - ly) * ((1.f - lx) * v00 + lx * v01) + ly * ((1.f - lx) * v10 + lx * v11);
  }
  mask[static_cast<long>(n) * npix + pix] = sigmoidf_(acc);
}

// ------------------------------------------------------------------------------------------------ post-processing (8f3)
// tensor2img (img_util.py:38-94): clamp[0,1] -> *255 -> round half-to-even -> uint8, RGB -> BGR, HWC; and the squared
// Y-channel difference against a ground-truth frame (metric_util.py:32-45, psnr_ssim.py:11-48), accumulated in double, one
// partial sum per block (deterministic, like ssim_y).  grid (blocks, batch), 256 threads.
__device__ __forceinline__ float y_of_u8(int b, int g, int r) {
  const double d = (static_cast<double>(static_cast<float>(b) / 255.f) * 24.966 + static_cast<double>(static_cast<float>(g) / 255.f) * 128.553) +
                   static_cast<double>(static_cast<float>(r) / 255.f) * 65.481 + 16.0;
  return static_cast<float>(d / 255.) * 255.f;
}
__global__ void __launch_bounds__(256) img_metrics_kernel(const float* __restrict__ sr, const float* __restrict__ gt, int H, int W,
                                                          uint8_t* __restrict__ bgr, double* __restrict__ sse) {
  const int n = blockIdx.y;
  const long npix = static_cast<long>(H) * W;
  const float* s = sr + static_cast<long>(n) * 3 * npix;
  const float* g = gt ? gt + static_cast<long>(n) * 3 * npix : nullptr;
  double acc = 0.0;
  for (long pix = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; pix < npix; pix += static_cast<long>(gridDim.x) * blockDim.x) {
    int q[3], qg[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      q[c] = unit_to_u8(s[c * npix + pix]);
      if (g) qg[c] = unit_to_u8(g[c * npix + pix]);
    }
    if (bgr) {
      uint8_t* o = bgr + (static_cast<long>(n) * npix + pix) * 3;
      o[0] = static_cast<uint8_t>(q[2]); o[1] = static_cast<uint8_t>(q[1]); o[2] = static_cast<uint8_t>(q[0]);
    }
    if (g) {
      const double d = static_cast<double>(y_of_u8(q[2], q[1], q[0])) - static_cast<double>(y_of_u8(qg[2], qg[1], qg[0]));
      acc += d * d;
    }
  }
  if (sse) {
    __shared__ double red[8];
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int i = 0; i < 8; ++i) t += red[i];
      sse[static_cast<long>(n) * gridDim.x + blockIdx.x] = t;   // one partial per block, summed by the caller in a fixed order: bit-reproducible
    }
  }
}

}  // namespace savsr

using namespace savsr;

// SSIM on the Y channel (psnr_ssim.py:85-129, _ssim 172-200; crop_border 0): both frames are quantised to the uint8 images
// tensor2img would produce, converted to the unrounded float32 Y of to_y_channel, and filtered in float64 with the 11x11
// Gaussian window (sigma 1.5) over the fully covered positions only.  Block = 16x16 map positions, the 26x26 Y patches of
// both frames in shared memory; one partial sum per block (deterministic), summed by the caller.
struct SsimParams {
  const float* sr;
  const float* gt;
  double* partials;
  int H, W, bx, by;
  double k[11];   // cv2.getGaussianKernel(11, 1.5); window = outer(k, k)
};
__global__ void __launch_bounds__(256) ssim_y_kernel(const __grid_constant__ SsimParams p) {
  __shared__ double y1[26][27], y2[26][27];
  __shared__ double red[8];
  const int n = blockIdx.z;
  const long npix = static_cast<long>(p.H) * p.W;
  const float* s = p.sr + static_cast<long>(n) * 3 * npix;
  const float* g = p.gt + static_cast<long>(n) * 3 * npix;
  const int oy0 = blockIdx.y * 16, ox0 = blockIdx.x * 16;
  for (int i = threadIdx.x; i < 26 * 26; i += 256) {
    const int r = i / 26, c = i - r * 26;
    const int y = oy0 + r, x = ox0 + c;
    double a = 0.0, b = 0.0;
    if (y < p.H && x < p.W) {
      const long pix = static_cast<long>(y) * p.W + x;
      int q[3], qg[3];
#pragma unroll
      for (int ch = 0; ch < 3; ++ch) {
        q[ch] = unit_to_u8(s[ch * npix + pix]);
        qg[ch] = unit_to_u8(g[ch * npix + pix]);
      }
      a = static_cast<double>(y_of_u8(q[2], q[1], q[0]));
      b = static_cast<double>(y_of_u8(qg[2], qg[1], qg[0]));
    }
    y1[r][c] = a; y2[r][c] = b;
  }
  __syncthreads();
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
  double val = 0.0;
  if (oy0 + ty < p.H - 10 && ox0 + tx < p.W - 10) {
    double mu1 = 0.0, mu2 = 0.0, s11 = 0.0, s22 = 0.0, s12 = 0.0;
    for (int i = 0; i < 11; ++i) {
#pragma unroll
      for (int j = 0; j < 11; ++j) {
        const double w = p.k[i] * p.k[j];
        const double a = y1[ty + i][tx + j], b = y2[ty + i][tx + j];
        mu1 += w * a; mu2 += w * b;
        s11 += w * (a * a); s22 += w * (b * b); s12 += w * (a * b);
      }
    }
    const double c1 = (0.01 * 255) * (0.01 * 255), c2 = (0.03 * 255) * (0.03 * 255);
    const double mu1_sq = mu1 * mu1, mu2_sq = mu2 * mu2, mu12 = mu1 * mu2;
    val = ((2 * mu12 + c1) * (2 * (s12 - mu12) + c2)) / ((mu1_sq + mu2_sq + c1) * ((s11 - mu1_sq) + (s22 - mu2_sq) + c2));
  }
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) val += __shfl_xor_sync(0xffffffffu, val, off);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = val;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < 8; ++i) t += red[i];
    p.partials[(static_cast<long>(n) * p.by + blockIdx.y) * p.bx + blockIdx.x] = t;
  }
}

template <class T>
static int pack_frames(const char* name, savsr_ctx* ctx, savsr_arena* arena, const T* x, int t, int h, int w, int dst_slot, savsr_stream st) {
  SAVSR_REQUIRE(ctx && arena && x, "%s: null pointer", name);
  DeviceGuard guard(ctx->device);
  SAVSR_REQUIRE(t >= 1 && 3 * t <= kC, "%s: %d frames do not fit 64 channels", name, t);
  SAVSR_REQUIRE(h >= 2 && w >= 2, "%s: LR frame %dx%d too small for reflect padding", name, h, w);
  SAVSR_REQUIRE(arena->height == h + (h & 1) && arena->width == w + (w & 1),
                "%s: arena %dx%d is not the even-padded size of %dx%d", name, arena->height, arena->width, h, w);
  SAVSR_REQUIRE(dst_slot >= 0 && dst_slot < arena->nslots, "%s: slot %d out of range", name, dst_slot);
  if (arena->batch == 0) return 0;
  const long npix = static_cast<long>(arena->height) * arena->width;
  const long total = arena->batch * npix * 8;
  const int blocks = static_cast<int>((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
  pack_frames_kernel<T><<<blocks, 256, 0, static_cast<cudaStream_t>(st)>>>(x, arena->base + static_cast<long>(dst_slot) * arena->batch * npix * kC,
                                                                          arena->batch, t, h, w, arena->height, arena->width, ctx->fmt);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int savsr_pack_frames(savsr_ctx* ctx, savsr_arena* arena, const float* x, int t, int h, int w, int dst_slot, savsr_stream st) {
  return pack_frames("savsr_pack_frames", ctx, arena, x, t, h, w, dst_slot, st);
}

extern "C" int savsr_pack_frames_u8(savsr_ctx* ctx, savsr_arena* arena, const uint8_t* x, int t, int h, int w, int dst_slot, savsr_stream st) {
  return pack_frames("savsr_pack_frames_u8", ctx, arena, x, t, h, w, dst_slot, st);
}

extern "C" int savsr_pack_frames_u8_table(savsr_ctx* ctx, savsr_arena* arena, const uint8_t* const* frames, int t, int h, int w, int dst_slot,
                                          savsr_stream st) {
  return pack_frames("savsr_pack_frames_u8_table", ctx, arena, frames, t, h, w, dst_slot, st);
}

extern "C" int savsr_pack_frames_u16_table(savsr_ctx* ctx, savsr_arena* arena, const uint16_t* const* frames, int t, int h, int w, int dst_slot,
                                           savsr_stream st) {
  return pack_frames("savsr_pack_frames_u16_table", ctx, arena, frames, t, h, w, dst_slot, st);
}

namespace savsr {
// The frame table is written by kernels whose by-value argument carries the pointers, never by a host-to-device copy: a copy from
// pageable host memory holds the host until the stream has drained, and between two forwards of a video that is an idle GPU.
struct FrameTableChunk {
  const uint8_t* ptrs[kFrameTableChunk];
};
__global__ void __launch_bounds__(kFrameTableChunk) write_frame_table_kernel(const __grid_constant__ FrameTableChunk c, const uint8_t** dst, int n) {
  if (static_cast<int>(threadIdx.x) < n) dst[threadIdx.x] = c.ptrs[threadIdx.x];
}
}  // namespace savsr

extern "C" int savsr_write_frame_table(savsr_ctx* ctx, const uint8_t** table_dev, const uint8_t* const* ptrs_host, int n, savsr_stream st) {
  SAVSR_REQUIRE(ctx && table_dev && ptrs_host && n >= 0, "savsr_write_frame_table: null pointer / negative count");
  for (int i = 0; i < n; ++i) SAVSR_REQUIRE(ptrs_host[i], "savsr_write_frame_table: frame pointer %d of %d is null", i, n);
  DeviceGuard guard(ctx->device);
  FrameTableChunk c = {};
  for (int i0 = 0; i0 < n; i0 += kFrameTableChunk) {
    const int m = n - i0 < kFrameTableChunk ? n - i0 : kFrameTableChunk;
    memcpy(c.ptrs, ptrs_host + i0, m * sizeof(c.ptrs[0]));
    write_frame_table_kernel<<<1, kFrameTableChunk, 0, static_cast<cudaStream_t>(st)>>>(c, table_dev + i0, m);
    SAVSR_CUDA(cudaGetLastError());
  }
  return 0;
}

namespace savsr {
// Pooling + the two scale_routing layers (no BatchNorm in them): shared by the inference prologue and the train-mode one (train_attn.cu).
int osa_prologue_front(savsr_ctx* ctx, const savsr_osa_params* convs, int nconvs, int batch, int npart, int npix, float inv_scale_h,
                       float inv_scale_w, cudaStream_t st) {
  OsaLaunch L;
  memset(&L, 0, sizeof(L));
  int max_ci = 0;
  for (int i = 0; i < nconvs; ++i) {
    L.c[i] = convs[i];
    max_ci = convs[i].ci > max_ci ? convs[i].ci : max_ci;
  }
  L.nconvs = nconvs; L.batch = batch; L.npart = npart; L.npix = npix;
  L.inv_h = inv_scale_h; L.inv_w = inv_scale_w;
  L.fmt = ctx->fmt;
  (void)launch_k(ctx->opt[SAVSR_OPT_PDL] != 0, osa_pool_kernel, dim3(max_ci / 64, batch, nconvs), dim3(kOsaThreads), 0, st, L);
  const int lin_split = batch >= 12 ? 3 : (batch >= 4 ? 2 : 1);
  const size_t lin_smem = static_cast<size_t>((batch + lin_split - 1) / lin_split) * 2 * max_ci * sizeof(float);
  SAVSR_REQUIRE(lin_smem <= 200 * 1024, "savsr_osa_prologue: batch %d too large for the routing kernel's shared memory", batch);
  if (lin_smem > 48 * 1024) {
    if (int rc = ensure_smem_attr(ctx, kAttrOsaLinear, osa_linear_kernel, 200 * 1024)) return rc;
  }
  (void)launch_k(ctx->opt[SAVSR_OPT_PDL] != 0, osa_linear_kernel, dim3((2 * max_ci + 7) / 8, nconvs, lin_split), dim3(256), lin_smem, st, L, 0);
  (void)launch_k(ctx->opt[SAVSR_OPT_PDL] != 0, osa_linear_kernel, dim3((max_ci + 7) / 8, nconvs, lin_split), dim3(256), lin_smem, st, L, 1);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}
}  // namespace savsr

extern "C" int savsr_osa_prologue(savsr_ctx* ctx, const savsr_osa_params* convs, int nconvs, int batch, int npart,
                                  int npix, float inv_scale_h, float inv_scale_w, savsr_stream st_) {
  SAVSR_REQUIRE(ctx && convs, "savsr_osa_prologue: null pointer");
  DeviceGuard guard(ctx->device);
  SAVSR_REQUIRE(nconvs >= 0 && nconvs <= kMaxOsa, "savsr_osa_prologue: nconvs %d out of range [0,%d]", nconvs, kMaxOsa);
  if (nconvs == 0 || batch == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(st_);
  OsaLaunch L;
  memset(&L, 0, sizeof(L));
  int max_ci = 0;
  for (int i = 0; i < nconvs; ++i) {
    const savsr_osa_params& c = convs[i];
    SAVSR_REQUIRE(c.ci > 0 && c.ci % 64 == 0 && c.ci <= 64 * SAVSR_MAX_SRC, "savsr_osa_prologue: conv %d ci %d unsupported", i, c.ci);
    SAVSR_REQUIRE(c.co == 64, "savsr_osa_prologue: conv %d co %d unsupported (64 only)", i, c.co);
    SAVSR_REQUIRE(c.att > 0 && c.att <= 32, "savsr_osa_prologue: conv %d attention channels %d out of range", i, c.att);
    SAVSR_REQUIRE(c.bank && c.r0_w && c.r0_b && c.r2_w && c.r2_b && c.fc_w && c.bn_scale && c.bn_shift && c.ch_w && c.ch_b &&
                  c.fl_w && c.fl_b && c.sp_w && c.sp_b && c.kn_w && c.kn_b && c.scratch && c.packed,
                  "savsr_osa_prologue: conv %d has a null parameter pointer", i);
    for (int s = 0; s < c.ci / 64; ++s) SAVSR_REQUIRE(c.pool[s], "savsr_osa_prologue: conv %d source %d has no pool buffer", i, s);
    L.c[i] = c;
    max_ci = c.ci > max_ci ? c.ci : max_ci;
  }
  L.nconvs = nconvs; L.batch = batch; L.npart = npart; L.npix = npix;
  L.inv_h = inv_scale_h; L.inv_w = inv_scale_w;
  L.fmt = ctx->fmt;
  if (int rc = osa_prologue_front(ctx, convs, nconvs, batch, npart, npix, inv_scale_h, inv_scale_w, st)) return rc;
  int asm_split = batch >= 16 ? 4 : (batch >= 6 ? 2 : 1);
  while ((batch + asm_split - 1) / asm_split > kAsmMaxSamples) ++asm_split;
  osa_assemble_kernel<<<dim3((64 * max_ci + 255) / 256, nconvs, asm_split), 256, 0, st>>>(L);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int savsr_ca_scale_residual(savsr_ctx* ctx, savsr_arena* arena, int t_slot, int x_slot, int dst_slot,
                                       const float* pool, int npart, const float* w1, const float* b1, const float* w2,
                                       const float* b2, float* y_scratch, savsr_stream st) {
  SAVSR_REQUIRE(ctx && arena && pool && w1 && b1 && w2 && b2 && y_scratch, "savsr_ca_scale_residual: null pointer");
  DeviceGuard guard(ctx->device);
  SAVSR_REQUIRE(t_slot >= 0 && t_slot < arena->nslots && x_slot >= 0 && x_slot < arena->nslots && dst_slot >= 0 &&
                dst_slot < arena->nslots, "savsr_ca_scale_residual: slot out of range");
  CaParams p;
  p.npix = static_cast<long>(arena->height) * arena->width;
  const long img = p.npix * kC * arena->batch;
  p.t = arena->base + t_slot * img;
  p.x = arena->base + x_slot * img;
  p.dst = arena->base + dst_slot * img;
  p.fmt = ctx->fmt; p.pool = pool; p.npart = npart; p.w1 = w1; p.b1 = b1; p.w2 = w2; p.b2 = b2; p.y = y_scratch;
  long blocks = (p.npix * 8 + 255) / 256;
  const long cap = 8L * ctx->sm_count / (arena->batch > 0 ? arena->batch : 1) + 1;
  if (blocks > cap) blocks = cap;
  if (arena->batch == 0) return 0;
  (void)launch_k(ctx->opt[SAVSR_OPT_PDL] != 0, ca_vector_kernel, dim3(arena->batch), dim3(1024), 0, static_cast<cudaStream_t>(st), p);
  (void)launch_k(ctx->opt[SAVSR_OPT_PDL] != 0, ca_scale_residual_kernel, dim3(static_cast<unsigned>(blocks), arena->batch), dim3(256), 0, static_cast<cudaStream_t>(st), p);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int savsr_osadapt_mask(savsr_ctx* ctx, const float* in16, int batch, int height, int width, const float* wa,
                                  const float* ba, const float* wb, const float* bb, const float* wc, const float* bc,
                                  float* half0, float* half1, float* mask, savsr_stream st_) {
  SAVSR_REQUIRE(ctx && in16 && wa && ba && wb && bb && wc && bc && half0 && half1 && mask, "savsr_osadapt_mask: null pointer");
  DeviceGuard guard(ctx->device);
  SAVSR_REQUIRE(height % 2 == 0 && width % 2 == 0, "savsr_osadapt_mask: size %dx%d must be even (pad_spatial)", height, width);
  if (batch == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(st_);
  const int h2 = height / 2, w2 = width / 2;
  const long npix2 = static_cast<long>(h2) * w2;
  dim3 g2(static_cast<unsigned>((npix2 + 63) / 64), batch);   // 256 threads = 64 half-resolution pixels x 4 channel quarters
  mask_conv16_kernel<true, false><<<g2, 256, 0, st>>>(in16, wa, ba, nullptr, half0, h2, w2);
  mask_conv16_kernel<false, true><<<g2, 256, 0, st>>>(half0, wb, bb, wc, half1, h2, w2);   // half1 <- the nine tap projections
  dim3 g1(static_cast<unsigned>((4 * npix2 + 255) / 256), batch);
  mask_final_kernel<<<g1, 256, 0, st>>>(half1, bc, mask, h2, w2);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

static long img_metrics_grid(const savsr_ctx* ctx, int height, int width) {
  const long npix = static_cast<long>(height) * width;
  long blocks = (npix + 255) / 256;
  if (blocks > 4L * ctx->sm_count) blocks = 4L * ctx->sm_count;
  return blocks;
}

extern "C" int savsr_img_metrics_blocks(const savsr_ctx* ctx, int height, int width) {
  return (ctx && height > 0 && width > 0) ? static_cast<int>(img_metrics_grid(ctx, height, width)) : 0;
}

extern "C" int savsr_img_metrics(savsr_ctx* ctx, const float* sr, const float* gt, int batch, int height, int width, uint8_t* bgr_u8,
                                 double* sse_y, savsr_stream st_) {
  SAVSR_REQUIRE(ctx && sr, "savsr_img_metrics: null pointer");
  DeviceGuard guard(ctx->device);
  SAVSR_REQUIRE(batch >= 0 && height > 0 && width > 0, "savsr_img_metrics: bad shape");
  SAVSR_REQUIRE(!sse_y || gt, "savsr_img_metrics: sse_y requested without a ground-truth frame");
  if (batch == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(st_);
  const long blocks = img_metrics_grid(ctx, height, width);
  img_metrics_kernel<<<dim3(static_cast<unsigned>(blocks), batch), 256, 0, st>>>(sr, gt, height, width, bgr_u8, sse_y);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int savsr_ssim_y_blocks(int height, int width) {
  if (height < 11 || width < 11) return 0;
  return ((height - 10 + 15) / 16) * ((width - 10 + 15) / 16);
}

extern "C" int savsr_ssim_y(savsr_ctx* ctx, const float* sr, const float* gt, int batch, int height, int width, double* partials,
                            savsr_stream st) {
  SAVSR_REQUIRE(ctx && sr && gt && partials, "savsr_ssim_y: null pointer");
  DeviceGuard guard(ctx->device);
  SAVSR_REQUIRE(batch >= 0 && height >= 11 && width >= 11, "savsr_ssim_y: frames of %dx%d are smaller than the 11x11 window", height, width);
  if (batch == 0) return 0;
  SsimParams p;
  p.sr = sr; p.gt = gt; p.partials = partials; p.H = height; p.W = width;
  p.bx = (width - 10 + 15) / 16; p.by = (height - 10 + 15) / 16;
  double sum = 0.0;
  for (int i = 0; i < 11; ++i) { p.k[i] = exp(-((i - 5.0) * (i - 5.0)) / (2.0 * 1.5 * 1.5)); sum += p.k[i]; }
  for (int i = 0; i < 11; ++i) p.k[i] /= sum;
  ssim_y_kernel<<<dim3(p.bx, p.by, batch), 256, 0, static_cast<cudaStream_t>(st)>>>(p);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}
