// SATU kernels (savsr_arch.py:217-376): bit-exact coordinate / index kernel + per-scale MLP table,
// spatio-temporal filtering, and the fused HR gather with the routed compress/expand experts.
//
// Coordinate arithmetic follows the reference's fp32 operation order exactly (CPU semantics: IEEE
// division by the scale, no FMA contraction), hence the explicit __fadd_rn/__fmul_rn/__fdiv_rn.
#include "common.cuh"

namespace savsr {

__device__ __forceinline__ float rel_q(int i, float s) { return __fdiv_rn(__fadd_rn(static_cast<float>(i), 0.5f), s); }
// R(i) = (q - floor(q + 1e-3)) - 0.5   (savsr_arch.py:331, 333)
__device__ __forceinline__ float rel_coord(int i, float s, int* cell) {
  const float q = rel_q(i, s);
  const float fl = floorf(__fadd_rn(q, 1e-3f));
  if (cell) *cell = static_cast<int>(fl);
  return __fsub_rn(__fsub_rn(q, fl), 0.5f);
}
// normalised base grid coordinate (savsr_arch.py:275-280), zero offset
__device__ __forceinline__ float base_norm(int i, float s, int n_lr) {
  float g = __fsub_rn(__fdiv_rn(__fadd_rn(static_cast<float>(i), 0.5f), s), 0.5f);
  g = __fsub_rn(__fdiv_rn(__fmul_rn(g, 2.f), static_cast<float>(n_lr - 1)), 1.f);
  return g;
}
// ATen grid_sampler un-normalisation, align_corners = True
__device__ __forceinline__ float unnormalize(float g, int n_lr) {
  return __fmul_rn(__fdiv_rn(__fadd_rn(g, 1.f), 2.f), static_cast<float>(n_lr - 1));
}

__host__ __device__ constexpr uint32_t desc_hi_1024() { return (1024u >> 4) | (1u << 14) | (2u << 29); }
__device__ __forceinline__ uint64_t make_desc64(uint32_t hi, uint32_t lo) { return (static_cast<uint64_t>(hi) << 32) | lo; }

__global__ void satu_axis_kernel(int n_out, int n_lr, float s, float* rel, int32_t* cell, float* base, int32_t* corner) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_out) return;
  int c;
  const float r = rel_coord(i, s, &c);
  if (rel) rel[i] = r;
  if (cell) cell[i] = c;
  const float g = base_norm(i, s, n_lr);
  if (base) base[i] = g;
  if (corner) corner[i] = static_cast<int32_t>(floorf(unnormalize(g, n_lr)));
}

// table[pix] = (offset_x, offset_y, st_offset_x, st_offset_y, r0..r3), the 4 -> 64 -> 64 MLP and its heads
// (savsr_arch.py:335-351).  One HR pixel per thread, weights in shared memory.
__global__ void __launch_bounds__(128) satu_table_kernel(const savsr_satu_weights wts, int H, int W, float s_h, float s_w,
                                                         float* __restrict__ table) {
  __shared__ __align__(16) float w0[4 * 64];    // [in][out]
  __shared__ __align__(16) float w2[64 * 64];   // [in][out]
  __shared__ __align__(16) float wh[8 * 64];    // [head][in]: offset(2), st_offset(2), routing(4)
  __shared__ float b0[64], b2[64], bh[8];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) w0[i] = wts.body0_w[(i & 63) * 4 + (i >> 6)];
  for (int i = threadIdx.x; i < 4096; i += blockDim.x) w2[i] = wts.body2_w[(i & 63) * 64 + (i >> 6)];
  for (int i = threadIdx.x; i < 512; i += blockDim.x) {
    const int hd = i >> 6, j = i & 63;
    wh[i] = hd < 2 ? wts.offset_w[hd * 64 + j] : hd < 4 ? wts.st_offset_w[(hd - 2) * 64 + j] : wts.routing_w[(hd - 4) * 64 + j];
  }
  if (threadIdx.x < 64) { b0[threadIdx.x] = wts.body0_b[threadIdx.x]; b2[threadIdx.x] = wts.body2_b[threadIdx.x]; }
  if (threadIdx.x < 8) {
    const int hd = threadIdx.x;
    bh[hd] = hd < 2 ? wts.offset_b[hd] : hd < 4 ? wts.st_offset_b[hd - 2] : wts.routing_b[hd - 4];
  }
  __syncthreads();
  const long pix = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  if (pix >= static_cast<long>(H) * W) return;
  const int i = pix / W, j = pix % W;
  float in[4];
  in[0] = __fdiv_rn(1.f, s_w);  // channel 0 is 1/s_w (savsr_arch.py:336)
  in[1] = __fdiv_rn(1.f, s_h);
  in[2] = rel_coord(i, s_h, nullptr);
  in[3] = rel_coord(j, s_w, nullptr);
  float e1[64];
#pragma unroll
  for (int o = 0; o < 64; ++o) {
    float a = b0[o];
#pragma unroll
    for (int k = 0; k < 4; ++k) a += w0[k * 64 + o] * in[k];
    e1[o] = fmaxf(a, 0.f);
  }
  float e2[64];
#pragma unroll
  for (int o = 0; o < 64; ++o) e2[o] = b2[o];
#pragma unroll 4
  for (int k = 0; k < 64; ++k) {
    const float a = e1[k];
    const float4* wr = reinterpret_cast<const float4*>(w2 + k * 64);
#pragma unroll
    for (int o4 = 0; o4 < 16; ++o4) {
      const float4 wv = wr[o4];
      e2[4 * o4 + 0] += a * wv.x; e2[4 * o4 + 1] += a * wv.y;
      e2[4 * o4 + 2] += a * wv.z; e2[4 * o4 + 3] += a * wv.w;
    }
  }
  float out[8];
#pragma unroll
  for (int hd = 0; hd < 8; ++hd) {
    float a = bh[hd];
#pragma unroll
    for (int k = 0; k < 64; ++k) a += wh[hd * 64 + k] * fmaxf(e2[k], 0.f);
    out[hd] = hd < 4 ? a : 1.f / (1.f + expf(-a));
  }
  float4* d = reinterpret_cast<float4*>(table + pix * 8);
  d[0] = make_float4(out[0], out[1], out[2], out[3]);
  d[1] = make_float4(out[4], out[5], out[6], out[7]);
}

// ------------------------------------------------------------------------------------------------ kernel_conv + sta_conv, fused
// sta[p][c] = sum_{t in 5x5} x[clamp(p + d_t)][c] * K_t[p][c],   K_t = LeakyReLU_0.1(W_t a[p] + b_t)   (savsr_arch.py:297-313)
// The unfused route materialises the 25 per-pixel kernels K_t (1600 channels, 83 MB per sample) and reads them back.  Here
// each tap is one M=128 (8x16-pixel tile) x N=64 x K=64 GEMM on tcgen05 whose accumulator is consumed straight from TMEM:
// the epilogue threads multiply it with the tap's neighbour feature (16-byte loads that hit L1) and keep the 25-tap sum
// in registers, so K never leaves the SM.  Work unit = batch of 2 tiles sharing one pass over the 25 weight blocks (8 KB each,
// streamed through a ring); TMEM holds 4 taps x 2 tiles of accumulators, so the tensor core runs up to 4 taps ahead.
// Warps: 0 = TMA producer, 1 = MMA issuer, 2..17 = epilogue (TMEM lane quadrant = warp % 4; 2 column halves x 2 tiles).
struct KstaParams {
  CUtensorMap tm_tile;            // box [64 ch, 8, 16, 1] over the LR arena
  const __nv_bfloat16* arena;
  const uint8_t* weights;         // packed [25][64][64], rows in SAVSR_ROWS_QUAD order
  const float* bias;              // [25][64]
  float slope;
  int batch, hp, wp, h, w;
  int a_slot, x_slot, dst_slot;
  int tiles_x, tiles_y;
  int nbatches, chunk;            // work items = 2-tile batches; `chunk` consecutive ones per CTA
  int fmt;
};
constexpr int kKstaThreads = 18 * 32;
constexpr int kKstaWStages = 6;
constexpr int kKstaSmem = 1024 + 4 * 16384 + kKstaWStages * 8192 + 512;

__global__ void __launch_bounds__(kKstaThreads, 1) satu_kconv_sta_kernel(const __grid_constant__ KstaParams p) {
  extern __shared__ uint8_t raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* smem_a = smem;                       // [2 buffers][2 tiles][16 KB]
  uint8_t* smem_w = smem + 4 * 16384;           // ring of weight blocks
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_w + kKstaWStages * 8192);
  uint64_t* a_full = bars;                      // [2]
  uint64_t* a_empty = a_full + 2;               // [2]
  uint64_t* w_full = a_empty + 2;               // [6]
  uint64_t* w_empty = w_full + kKstaWStages;    // [6]
  uint64_t* t_full = w_empty + kKstaWStages;    // [8]  accumulator (tap & 3) * 2 + tile
  uint64_t* t_empty = t_full + 8;               // [8]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles = p.tiles_x * p.tiles_y;
  const int per_img = (tiles + 1) >> 1;          // 2-tile batches per sample (the last one may hold a single tile)
  const int item_begin = blockIdx.x * p.chunk;
  const int item_end = min(item_begin + p.chunk, p.nbatches);

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&p.tm_tile);
    for (int i = 0; i < 2; ++i) { mbar_init(a_full + i, 1); mbar_init(a_empty + i, 1); }
    for (int i = 0; i < kKstaWStages; ++i) { mbar_init(w_full + i, 1); mbar_init(w_empty + i, 1); }
    for (int i = 0; i < 8; ++i) { mbar_init(t_full + i, 1); mbar_init(t_empty + i, 8); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================================ producer ================================
    if (lane == 0) {
      int ws = 0, wph = 0;
      for (int item = item_begin, it = 0; item < item_end; ++item, ++it) {
        const int n = item / per_img, t0 = (item - n * per_img) * 2;
        const int cnt = min(2, tiles - t0);
        const int ab = it & 1;
        mbar_wait(a_empty + ab, ((it >> 1) & 1) ^ 1);
        mbar_expect_tx(a_full + ab, cnt * 16384u);
        for (int j = 0; j < cnt; ++j) {
          const int tj = t0 + j, ty = tj / p.tiles_x, tx = tj - ty * p.tiles_x;
          tma_load_4d(smem_a + (ab * 2 + j) * 16384, &p.tm_tile, a_full + ab, 0, tx * kTileW, ty * kTileH, p.a_slot * p.batch + n);
        }
        for (int tap = 0; tap < 25; ++tap) {
          mbar_wait(w_empty + ws, wph ^ 1);
          mbar_expect_tx(w_full + ws, 8192u);
          bulk_load(smem_w + ws * 8192, p.weights + tap * 8192, 8192u, w_full + ws);
          if (++ws == kKstaWStages) { ws = 0; wph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ================================
    const uint32_t idesc = umma_idesc_f16(64, p.fmt);
    constexpr uint32_t hi = desc_hi_1024();
    const uint32_t a_lo0 = (smem_u32(smem_a) >> 4) & 0x3fffu, w_lo0 = (smem_u32(smem_w) >> 4) & 0x3fffu;
    int ws = 0, wph = 0;
    uint32_t use_bits = 0;
    for (int item = item_begin, it = 0; item < item_end; ++item, ++it) {
      const int n = item / per_img, t0 = (item - n * per_img) * 2;
      const int cnt = min(2, tiles - t0);
      const int ab = it & 1;
      mbar_wait(a_full + ab, (it >> 1) & 1);
      tc_fence_after();
      for (int tap = 0; tap < 25; ++tap) {
        mbar_wait(w_full + ws, wph);
        tc_fence_after();
        const uint32_t wl = w_lo0 + ws * (8192 >> 4);
        for (int j = 0; j < cnt; ++j) {
          const int acc = (tap & 3) * 2 + j;
          mbar_wait(t_empty + acc, ((use_bits >> acc) & 1u) ^ 1u);
          use_bits ^= 1u << acc;
          tc_fence_after();
          const uint32_t al = a_lo0 + (ab * 2 + j) * (16384 >> 4);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16(tmem_base + acc * 64, make_desc64(hi, al + 2 * k), make_desc64(hi, wl + 2 * k), idesc, k ? 1u : 0u);
            umma_commit(t_full + acc);
          }
          __syncwarp();
        }
        if (elect_one()) umma_commit(w_empty + ws);
        __syncwarp();
        if (++ws == kKstaWStages) { ws = 0; wph ^= 1; }
      }
      if (elect_one()) umma_commit(a_empty + ab);
      __syncwarp();
    }
  } else {
    // ================================ epilogue ================================
    const int quad = warp & 3;
    const int r = (warp - 2) >> 2;
    const int half = r & 1, tj = r >> 1;
    const int g = lane >> 2, q = lane & 3;
    const int ch0 = half * 32 + q * 8;
    const long npix = static_cast<long>(p.hp) * p.wp;
    const float slope = p.slope;
    uint32_t use_bits = 0;
    for (int item = item_begin; item < item_end; ++item) {
      const int n = item / per_img, t0 = (item - n * per_img) * 2;
      const int cnt = min(2, tiles - t0);
      if (tj >= cnt) continue;   // single-tile batch: the accumulators of tile 1 are not touched, their phases stay put
      const int tile = t0 + tj, ty = tile / p.tiles_x, tx = tile - ty * p.tiles_x;
      const int px = tx * kTileW + g;
      const int py0 = ty * kTileH + quad * 4;
      const __nv_bfloat16* xs = p.arena + (static_cast<long>(p.x_slot) * p.batch + n) * npix * kC + ch0;
      float acc[4][8];
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[j][i] = 0.f;
      for (int tap = 0; tap < 25; ++tap) {
        const int a = (tap & 3) * 2 + tj;
        const int dy = tap / 5 - 2, dx = tap - (tap / 5) * 5 - 2;
        // neighbour features first: their latency hides behind the accumulator wait
        const int sx = min(max(px + dx, 0), p.w - 1);
        uint4 nb[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int sy = min(max(py0 + j + dy, 0), p.h - 1);
          nb[j] = __ldg(reinterpret_cast<const uint4*>(xs + (static_cast<long>(sy) * p.wp + sx) * kC));
        }
        const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + tap * 64 + ch0));
        const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + tap * 64 + ch0) + 1);
        const float bias[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
        mbar_wait(t_full + a, (use_bits >> a) & 1u);
        use_bits ^= 1u << a;
        tc_fence_after();
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + static_cast<uint32_t>(a * 64 + half * 32);
        uint32_t ra[16], rb[16];
        tmem_ld_16x256b_x4(taddr, ra);
        tmem_ld_16x256b_x4(taddr + (16u << 16), rb);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(t_empty + a);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int i = 2 * k + (e & 1);
            {
              const float t = __uint_as_float(ra[4 * k + e]) + bias[i];
              const float kv = fmaxf(t, slope * t);   // LeakyReLU for 0 <= slope <= 1
              const uint32_t w32 = i < 2 ? nb[e >> 1].x : i < 4 ? nb[e >> 1].y : i < 6 ? nb[e >> 1].z : nb[e >> 1].w;
              acc[e >> 1][i] += kv * ((i & 1) ? h_hi(w32, p.fmt) : h_lo(w32, p.fmt));
            }
            {
              const float t = __uint_as_float(rb[4 * k + e]) + bias[i];
              const float kv = fmaxf(t, slope * t);
              const uint32_t w32 = i < 2 ? nb[2 + (e >> 1)].x : i < 4 ? nb[2 + (e >> 1)].y : i < 6 ? nb[2 + (e >> 1)].z : nb[2 + (e >> 1)].w;
              acc[2 + (e >> 1)][i] += kv * ((i & 1) ? h_hi(w32, p.fmt) : h_lo(w32, p.fmt));
            }
          }
        }
      }
      // zeros outside the unpadded h x w region (like the unfused kernel); nothing outside the arena
      __nv_bfloat16* d = const_cast<__nv_bfloat16*>(p.arena) + (static_cast<long>(p.dst_slot) * p.batch + n) * npix * kC + ch0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int py = py0 + j;
        if (px < p.wp && py < p.hp) {
          const bool in = px < p.w && py < p.h;
          uint4 u;
          u.x = in ? pack_h2(acc[j][0], acc[j][1], p.fmt) : 0u;
          u.y = in ? pack_h2(acc[j][2], acc[j][3], p.fmt) : 0u;
          u.z = in ? pack_h2(acc[j][4], acc[j][5], p.fmt) : 0u;
          u.w = in ? pack_h2(acc[j][6], acc[j][7], p.fmt) : 0u;
          *reinterpret_cast<uint4*>(d + (static_cast<long>(py) * p.wp + px) * kC) = u;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------ operand-tile helpers
__device__ __forceinline__ uint4 pack8(const float (&a)[8], int fmt) {
  uint4 o;
  o.x = pack_h2(a[0], a[1], fmt); o.y = pack_h2(a[2], a[3], fmt); o.z = pack_h2(a[4], a[5], fmt); o.w = pack_h2(a[6], a[7], fmt);
  return o;
}
// byte offset of 16-byte chunk `c` of row `r` in a [rows][128 B] SWIZZLE_128B tile
__device__ __forceinline__ int swz(int r, int c) { return r * 128 + ((c ^ (r & 7)) << 4); }

// ------------------------------------------------------------------------------------------------ HR stage, one kernel
// Everything of SATU at HR resolution and the tail, without any HR-resolution intermediate in memory
// (savsr_arch.py:344-376 STAUpsample.forward from the gathers on, 738-739 tail + bilinear skip):
//
//   F = bilinear gather of x at base + offset, S = bilinear gather of sta at base + st_offset   (zeros padding, align_corners)
//   U = F Wc^T (4 experts' compress matrices stacked) ; V[e*8+k] = r_e * sum_e' r_e' U[e'*8+k]  (routing, per pixel)
//   fea = V We^T + F ; Y = [S | fea] Wf^T + bf ; sr = conv3x3(Y; Wt) + bt + bilinear(x_center)
//
// Between the gathers and the output everything is LINEAR given V, so fusion and tail are composed on the host:
//   Z[q][tap*3+c] = S[q] Wcs^T + F[q] Wcf^T + V[q] Wv^T + zb ,   Wcs|Wcf = Wt_tap Wf ,  Wv = Wcf We ,  zb = Wt_tap bf
//   sr[p][c] = bt[c] + sum_tap Z[p + d_tap][tap*3+c]   over the taps whose pixel p + d_tap lies inside the image
// i.e. per HR pixel 27 partial products instead of a 64-channel feature, summed over the 3x3 neighbourhood from shared memory.
// A CTA owns a 32 x 13 block of HR pixels; it evaluates Z on the 34 x 15 ringed block (510 pixels = 4 M-tiles of 128, 1.23x
// recompute) and loops over the samples of the batch with the sample-independent sampling corners of the block cached in smem.
//
// Warp roles (17 warps):   9..16  gather: build the F and S operand tiles (16-bit, 128-byte swizzled K-major) in a 2-stage ring
//                          8      MMA issuer (tcgen05, accumulators U and Z in TMEM, double buffered)
//                          0..7   consumers, two groups alternating tiles: routing (U -> V tile), Z -> smem, and, once per
//                                 block and sample, the 9-tap sum + bias + bilinear skip -> fp32 NCHW stores (128 B per warp row)
//
// I/O modes (template U8): fp32 (the module's forward contract) reads the skip from the fp32 window and stores fp32 NCHW; 8-bit reads it
// from the uint8 BGR window [batch][t][h][w][3] through the same u / 255 as the first layer, so the skip is the same fp32 number, and
// stores tensor2img's uint8 HWC BGR [batch][H][W][3] of the same fp32 value the fp32 mode would have written.
struct HrParams {
  const __nv_bfloat16* lr;
  const float* table;        // [H*W][8]: offset x,y | st_offset x,y | r0..r3
  const float* base_y;
  const float* base_x;
  const uint8_t* weights;    // 4 x [32 rows][128 B] K-major swizzled: Wc (rows e*8+k) | Wcf | Wcs | Wv (K = 32), rows of Wcf/Wcs/Wv = tap*3+c
  const float* zbias;        // [32]: zb[tap*3+c], 27 used
  const float* tail_bias;    // [3]
  const void* x_in;          // bilinear skip of the centre frame: fp32 [batch][t][3][h][w], or uint8 BGR [batch][t][h][w][3]
  void* out;                 // fp32 [batch][3][H][W], or uint8 BGR [batch][H][W][3]
  int batch, hp, wp, h, w, H, W;
  int x_slot, sta_slot;
  int t, centre;
  int regions_x, nregions;
  int fmt;
};

constexpr int kHrRW = 32, kHrRH = 13;                  // interior block
constexpr int kHrPW = kHrRW + 2, kHrPH = kHrRH + 2;    // ringed block 34 x 15 = 510 pixels
constexpr int kHrPix = 512;                            // 4 M-tiles
constexpr int kHrTiles = 4;
constexpr int kHrConsumerWarps = 8, kHrGatherWarps = 16;
constexpr int kHrIssuerWarp = kHrConsumerWarps;
constexpr int kHrThreads = 32 * (kHrConsumerWarps + 1 + kHrGatherWarps);
constexpr int kHrStages = 2;
constexpr int kHrZK = 27;
// shared-memory map (bytes from the 1024-aligned base)
constexpr int kHrOffFS = 0;                                    // [stages][F 16 KB | S 16 KB]
constexpr int kHrOffV = kHrOffFS + kHrStages * 32768;          // [2][16 KB]
constexpr int kHrOffW = kHrOffV + 2 * 16384;                   // 16 KB
constexpr int kHrOffZ = kHrOffW + 16384;                       // __half [2 buffers][27][512]: partial products of two (block, sample) pairs
constexpr int kHrOffCO = kHrOffZ + 2 * kHrZK * kHrPix * 2;     // uint4 [2][512]: element offsets of the four corner pixels inside the LR image
constexpr int kHrOffCW = kHrOffCO + 2 * kHrPix * 16;           // uint2 [2][512]: the four bilinear weights as 16-bit pairs (w00 w01 | w10 w11), 0 = outside
constexpr int kHrOffBar = kHrOffCW + 2 * kHrPix * 8;
constexpr int kHrSmem = 1024 + kHrOffBar + 512;   // 16 mbarriers, the TMEM slot, zbias[32]

// Packed 16-bit arithmetic of the gather: out = sum_q w_q * v_q on two channels at a time (HFMA2), in the operand format itself.
// The result feeds the tensor core as a 16-bit operand anyway; accumulating the four corners in that format costs about one
// extra rounding and needs 4x fewer instructions than convert + fp32 FMA + convert back (the gather is instruction-bound).
template <int FMT> struct Pk;
template <> struct Pk<SAVSR_FMT_BF16> {
  using T2 = __nv_bfloat162;
  static __device__ __forceinline__ uint32_t pair(float a, float b) { T2 r = __floats2bfloat162_rn(a, b); return *reinterpret_cast<uint32_t*>(&r); }
  static __device__ __forceinline__ T2 lo(uint32_t w) { return __low2bfloat162(*reinterpret_cast<T2*>(&w)); }
  static __device__ __forceinline__ T2 hi(uint32_t w) { return __high2bfloat162(*reinterpret_cast<T2*>(&w)); }
};
template <> struct Pk<SAVSR_FMT_FP16> {
  using T2 = __half2;
  static __device__ __forceinline__ uint32_t pair(float a, float b) { T2 r = __floats2half2_rn(a, b); return *reinterpret_cast<uint32_t*>(&r); }
  static __device__ __forceinline__ T2 lo(uint32_t w) { return __low2half2(*reinterpret_cast<T2*>(&w)); }
  static __device__ __forceinline__ T2 hi(uint32_t w) { return __high2half2(*reinterpret_cast<T2*>(&w)); }
};
template <int FMT>
__device__ __forceinline__ uint32_t pk_mul(uint32_t v, typename Pk<FMT>::T2 w) {
  typename Pk<FMT>::T2 r = __hmul2(*reinterpret_cast<typename Pk<FMT>::T2*>(&v), w);
  return *reinterpret_cast<uint32_t*>(&r);
}
template <int FMT>
__device__ __forceinline__ uint32_t pk_fma(uint32_t v, typename Pk<FMT>::T2 w, uint32_t acc) {
  typename Pk<FMT>::T2 r = __hfma2(*reinterpret_cast<typename Pk<FMT>::T2*>(&v), w, *reinterpret_cast<typename Pk<FMT>::T2*>(&acc));
  return *reinterpret_cast<uint32_t*>(&r);
}
template <int FMT>
__device__ __forceinline__ uint4 pk_blend(const uint4 (&v)[4], uint2 w) {
  const typename Pk<FMT>::T2 w0 = Pk<FMT>::lo(w.x), w1 = Pk<FMT>::hi(w.x), w2 = Pk<FMT>::lo(w.y), w3 = Pk<FMT>::hi(w.y);
  uint4 a;
  a.x = pk_mul<FMT>(v[0].x, w0); a.y = pk_mul<FMT>(v[0].y, w0); a.z = pk_mul<FMT>(v[0].z, w0); a.w = pk_mul<FMT>(v[0].w, w0);
  a.x = pk_fma<FMT>(v[1].x, w1, a.x); a.y = pk_fma<FMT>(v[1].y, w1, a.y); a.z = pk_fma<FMT>(v[1].z, w1, a.z); a.w = pk_fma<FMT>(v[1].w, w1, a.w);
  a.x = pk_fma<FMT>(v[2].x, w2, a.x); a.y = pk_fma<FMT>(v[2].y, w2, a.y); a.z = pk_fma<FMT>(v[2].z, w2, a.z); a.w = pk_fma<FMT>(v[2].w, w2, a.w);
  a.x = pk_fma<FMT>(v[3].x, w3, a.x); a.y = pk_fma<FMT>(v[3].y, w3, a.y); a.z = pk_fma<FMT>(v[3].z, w3, a.z); a.w = pk_fma<FMT>(v[3].w, w3, a.w);
  return a;
}

// ATen upsample_bilinear2d (align_corners = False) source index / weight with the size ratio precomputed by the caller.
__device__ __forceinline__ void bilinear_src_scaled(int dst, float scale, int in_size, int& i0, int& i1, float& l1) {
  float src = scale * (static_cast<float>(dst) + 0.5f) - 0.5f;
  src = src < 0.f ? 0.f : src;
  i0 = static_cast<int>(src);
  i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
  l1 = src - static_cast<float>(i0);
}

template <int FMT, bool U8>
__global__ void __launch_bounds__(kHrThreads, 1) satu_hr_kernel(const __grid_constant__ HrParams p) {
  extern __shared__ uint8_t raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* sFS = smem + kHrOffFS;
  uint8_t* sV = smem + kHrOffV;
  uint8_t* sW = smem + kHrOffW;
  __half* sZ = reinterpret_cast<__half*>(smem + kHrOffZ);
  uint4* sCO = reinterpret_cast<uint4*>(smem + kHrOffCO);
  uint2* sCW = reinterpret_cast<uint2*>(smem + kHrOffCW);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kHrOffBar);
  uint64_t* fs_full = bars;            // [2]  gather warps -> issuer
  uint64_t* fs_empty = bars + 2;       // [2]  issuer (commit) -> gather warps
  uint64_t* u_full = bars + 4;         // [2]  issuer (commit) -> consumers
  uint64_t* v_full = bars + 6;         // [2]  consumers -> issuer
  uint64_t* z_full = bars + 8;         // [2]  issuer (commit) -> consumers
  uint64_t* acc_empty = bars + 10;     // [2]  consumers -> issuer: U / Z accumulators of the buffer are free again
  uint64_t* zb_full = bars + 12;       // [2]  consumers -> gather warps: all 27 x 510 partial products of a (block, sample) are in shared memory
  uint64_t* zb_empty = bars + 14;      // [2]  gather warps -> consumers: that buffer has been summed and may be overwritten
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < 16384 / 16; i += kHrThreads) *reinterpret_cast<uint4*>(sW + i * 16) = __ldg(reinterpret_cast<const uint4*>(p.weights) + i);
  if (tid == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(fs_full + i, kHrGatherWarps); mbar_init(fs_empty + i, 1); mbar_init(u_full + i, 1);
      mbar_init(v_full + i, 4); mbar_init(z_full + i, 1); mbar_init(acc_empty + i, 4);
      mbar_init(zb_full + i, 4 * kHrTiles); mbar_init(zb_empty + i, kHrGatherWarps);
    }
    fence_barrier_init();
  }
  if (warp == kHrIssuerWarp) tmem_alloc<128>(tmem_slot);
  if (tid < 32) reinterpret_cast<float*>(tmem_slot + 4)[tid] = __ldg(p.zbias + tid);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tm = *tmem_slot;                  // columns: U0 [0,32) Z0 [32,64) U1 [64,96) Z1 [96,128)
  const long NPIX = static_cast<long>(p.H) * p.W;
  const long lr_img = static_cast<long>(p.hp) * p.wp * kC;

  if (warp > kHrIssuerWarp) {
    // ================================ gather warps (operand producers + the 9-tap tail) ================================
    const int gtid = tid - 32 * (kHrIssuerWarp + 1);
    constexpr int kGT = 32 * kHrGatherWarps;
    const float wm1 = static_cast<float>(p.w - 1), hm1 = static_cast<float>(p.h - 1);
    const float sk_sy = static_cast<float>(p.h) / static_cast<float>(p.H), sk_sx = static_cast<float>(p.w) / static_cast<float>(p.W);
    const int plane = p.h * p.w;
    const float bt0 = __ldg(p.tail_bias), bt1 = __ldg(p.tail_bias + 1), bt2 = __ldg(p.tail_bias + 2);
    uint32_t it = 0, rn = 0;                     // running tile / (block, sample) counters of this CTA
    int prevY0 = 0, prevX0 = 0, prevN = -1;      // the (block, sample) whose partial products are summed next

    // sr[p][c] = bt[c] + sum over the 3x3 taps inside the image of Z[p + d_tap][tap*3+c] + bilinear skip; one HR pixel per thread
    auto tail = [&](uint32_t k, int Y0, int X0, int n) {
      const int zb = k & 1;
      mbar_wait(zb_full + zb, (k >> 1) & 1u);
      const __half* z0 = sZ + zb * (kHrZK * kHrPix);
      if (gtid < kHrRW * kHrRH) {
        const int iy = gtid >> 5, ix = gtid & 31;
        const int Y = Y0 + 1 + iy, X = X0 + 1 + ix;
        if (Y < p.H && X < p.W) {
          int y0, y1, x0, x1;
          float ly, lx;
          bilinear_src_scaled(Y, sk_sy, p.h, y0, y1, ly);
          bilinear_src_scaled(X, sk_sx, p.w, x0, x1, lx);
          const long xc = static_cast<long>(n * p.t + p.centre) * 3 * plane;   // centre frame of sample n (elements, either layout)
          const int o00 = y0 * p.w + x0, o01 = y0 * p.w + x1, o10 = y1 * p.w + x0, o11 = y1 * p.w + x1;
          float sk[3];
#pragma unroll
          for (int ch = 0; ch < 3; ++ch) {
            float a, bb, cc, d;
            if constexpr (U8) {
              const uint8_t* pl = static_cast<const uint8_t*>(p.x_in) + xc + 2 - ch;
              a = u8_to_unit(__ldg(pl + 3 * o00)); bb = u8_to_unit(__ldg(pl + 3 * o01));
              cc = u8_to_unit(__ldg(pl + 3 * o10)); d = u8_to_unit(__ldg(pl + 3 * o11));
            } else {
              const float* pl = static_cast<const float*>(p.x_in) + xc + ch * plane;
              a = __ldg(pl + o00); bb = __ldg(pl + o01); cc = __ldg(pl + o10); d = __ldg(pl + o11);
            }
            sk[ch] = (1.f - ly) * ((1.f - lx) * a + lx * bb) + ly * ((1.f - lx) * cc + lx * d);
          }
          float acc0 = bt0, acc1 = bt1, acc2 = bt2;
#pragma unroll
          for (int dy = 0; dy < 3; ++dy) {
            const bool vy = static_cast<unsigned>(Y + dy - 1) < static_cast<unsigned>(p.H);
#pragma unroll
            for (int dx = 0; dx < 3; ++dx) {
              const bool v = vy && static_cast<unsigned>(X + dx - 1) < static_cast<unsigned>(p.W);
              const __half* z = z0 + ((dy * 3 + dx) * 3) * kHrPix + (iy + dy) * kHrPW + ix + dx;
              acc0 += v ? __half2float(z[0]) : 0.f;
              acc1 += v ? __half2float(z[kHrPix]) : 0.f;
              acc2 += v ? __half2float(z[2 * kHrPix]) : 0.f;
            }
          }
          if constexpr (U8) {
            // 3 bytes per pixel: W * 3 has any alignment, so plain byte stores (a warp row is 96 contiguous bytes)
            uint8_t* o = static_cast<uint8_t*>(p.out) + (static_cast<long>(n) * NPIX + static_cast<long>(Y) * p.W + X) * 3;
            o[0] = static_cast<uint8_t>(unit_to_u8(acc2 + sk[2])); o[1] = static_cast<uint8_t>(unit_to_u8(acc1 + sk[1]));
            o[2] = static_cast<uint8_t>(unit_to_u8(acc0 + sk[0]));
          } else {
            float* o = static_cast<float*>(p.out) + static_cast<long>(n) * 3 * NPIX + static_cast<long>(Y) * p.W + X;
            o[0] = acc0 + sk[0]; o[NPIX] = acc1 + sk[1]; o[2 * NPIX] = acc2 + sk[2];
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(zb_empty + zb);
    };

    for (int r = blockIdx.x; r < p.nregions; r += gridDim.x) {
      const int Y0 = (r / p.regions_x) * kHrRH - 1, X0 = (r % p.regions_x) * kHrRW - 1;   // origin of the ringed block
      named_barrier(2, kGT);             // every gather warp is done reading the previous block's corners
      for (int i = gtid; i < kHrPix; i += kGT) {
        const int py = i / kHrPW, px = i - py * kHrPW;
        const int Y = Y0 + py, X = X0 + px;
        uint4 co[2] = {make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0)};
        uint2 cw[2] = {make_uint2(0, 0), make_uint2(0, 0)};
        if (i < kHrPW * kHrPH && Y >= 0 && Y < p.H && X >= 0 && X < p.W) {
          const float4 t0 = __ldg(reinterpret_cast<const float4*>(p.table + (static_cast<long>(Y) * p.W + X) * 8));
          const float bx = __ldg(p.base_x + X), by = __ldg(p.base_y + Y);
          const float off[2][2] = {{t0.x, t0.y}, {t0.z, t0.w}};
#pragma unroll
          for (int s = 0; s < 2; ++s) {
            // grid = base + offset * 2 / (n - 1) (savsr_arch.py:285-287), then ATen's align_corners un-normalisation
            const float gx = __fadd_rn(bx, __fdiv_rn(__fmul_rn(off[s][0], 2.f), wm1));
            const float gy = __fadd_rn(by, __fdiv_rn(__fmul_rn(off[s][1], 2.f), hm1));
            const float ix = unnormalize(gx, p.w), iy = unnormalize(gy, p.h);
            const float x0f = floorf(ix), y0f = floorf(iy);
            const int x0 = static_cast<int>(x0f), y0 = static_cast<int>(y0f);
            const float tx = ix - x0f, ty = iy - y0f;
            const bool vx0 = x0 >= 0 && x0 < p.w, vx1 = x0 + 1 >= 0 && x0 + 1 < p.w;
            const bool vy0 = y0 >= 0 && y0 < p.h, vy1 = y0 + 1 >= 0 && y0 + 1 < p.h;
            const int xa = vx0 ? x0 : 0, xb = vx1 ? x0 + 1 : 0, ya = (vy0 ? y0 : 0) * p.wp, yb = (vy1 ? y0 + 1 : 0) * p.wp;
            const float wx0 = vx0 ? 1.f - tx : 0.f, wx1 = vx1 ? tx : 0.f, wy0 = vy0 ? 1.f - ty : 0.f, wy1 = vy1 ? ty : 0.f;
            co[s] = make_uint4((ya + xa) * kC, (ya + xb) * kC, (yb + xa) * kC, (yb + xb) * kC);
            cw[s] = make_uint2(Pk<FMT>::pair(wy0 * wx0, wy0 * wx1), Pk<FMT>::pair(wy1 * wx0, wy1 * wx1));
          }
        }
        sCO[i] = co[0]; sCO[kHrPix + i] = co[1];
        sCW[i] = cw[0]; sCW[kHrPix + i] = cw[1];
      }
      named_barrier(2, kGT);
      for (int n = 0; n < p.batch; ++n, ++rn) {
        const __nv_bfloat16* img0 = p.lr + (static_cast<long>(p.x_slot) * p.batch + n) * lr_img;
        const __nv_bfloat16* img1 = p.lr + (static_cast<long>(p.sta_slot) * p.batch + n) * lr_img;
        for (int t = 0; t < kHrTiles; ++t, ++it) {
          const int stage = it & 1;
          mbar_wait(fs_empty + stage, ((it >> 1) & 1u) ^ 1u);
          uint8_t* dst = sFS + stage * 32768;
#pragma unroll 1
          for (int id = gtid; id < 128 * 8; id += kGT) {
            const int lp = id >> 3, chunk = id & 7;
            const int i = t * 128 + lp;
            const uint4 c0 = sCO[i], c1 = sCO[kHrPix + i];
            const uint2 w0 = sCW[i], w1 = sCW[kHrPix + i];
            const __nv_bfloat16* b0 = img0 + chunk * 8;
            const __nv_bfloat16* b1 = img1 + chunk * 8;
            uint4 v0[4], v1[4];
            v0[0] = __ldg(reinterpret_cast<const uint4*>(b0 + c0.x)); v0[1] = __ldg(reinterpret_cast<const uint4*>(b0 + c0.y));
            v0[2] = __ldg(reinterpret_cast<const uint4*>(b0 + c0.z)); v0[3] = __ldg(reinterpret_cast<const uint4*>(b0 + c0.w));
            v1[0] = __ldg(reinterpret_cast<const uint4*>(b1 + c1.x)); v1[1] = __ldg(reinterpret_cast<const uint4*>(b1 + c1.y));
            v1[2] = __ldg(reinterpret_cast<const uint4*>(b1 + c1.z)); v1[3] = __ldg(reinterpret_cast<const uint4*>(b1 + c1.w));
            const int so = swz(lp, chunk);
            *reinterpret_cast<uint4*>(dst + so) = pk_blend<FMT>(v0, w0);
            *reinterpret_cast<uint4*>(dst + 16384 + so) = pk_blend<FMT>(v1, w1);
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive(fs_full + stage);
        }
        // the previous (block, sample) has long been through the tensor core by now: sum its taps while this one's tiles drain
        if (prevN >= 0) tail(rn - 1, prevY0, prevX0, prevN);
        prevY0 = Y0; prevX0 = X0; prevN = n;
      }
    }
    if (prevN >= 0) tail(rn - 1, prevY0, prevX0, prevN);
  } else if (warp == kHrIssuerWarp) {
    // ================================ MMA issuer (warp-uniform control flow, elected issue) ================================
    constexpr uint32_t hi = desc_hi_1024();
    const uint32_t idesc = umma_idesc_f16(32, FMT), idesc64 = umma_idesc_f16(64, FMT);
    const uint32_t loFS = (smem_u32(sFS) >> 4) & 0x3fff, loV = (smem_u32(sV) >> 4) & 0x3fff, loW = (smem_u32(sW) >> 4) & 0x3fff;
    const uint32_t loWc = loW, loWcs = loW + (8192 >> 4), loWv = loW + (12288 >> 4);    // Wcf sits right behind Wc (rows 32..63 of the N = 64 tile)
    int total = 0;
    for (int r = blockIdx.x; r < p.nregions; r += gridDim.x) total += p.batch * kHrTiles;
    for (int it = 0; it <= total; ++it) {
      if (it > 0) {
        // second GEMM of the previous tile: Z += V Wv^T (K = 32), as soon as the consumers have written its V tile
        const int pb = (it - 1) & 1;
        mbar_wait(v_full + pb, ((it - 1) >> 1) & 1u);
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 2; ++k)
            umma_bf16(tm + pb * 64 + 32, make_desc64(hi, loV + pb * (16384 >> 4) + 2 * k), make_desc64(hi, loWv + 2 * k), idesc, 1u);
          umma_commit(z_full + pb);
        }
        __syncwarp();
      }
      if (it == total) break;
      const int b = it & 1;           // stage of the F/S ring == accumulator buffer
      mbar_wait(fs_full + b, (it >> 1) & 1u);
      mbar_wait(acc_empty + b, ((it >> 1) & 1u) ^ 1u);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t loF = loFS + b * (32768 >> 4), loS = loF + (16384 >> 4);
        // [U | Z] = F [Wc ; Wcf]^T in ONE N = 64 chain (the two weight tiles are adjacent in shared memory and U, Z adjacent in
        // TMEM), so the F tile is read once; then Z += S Wcs^T
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_bf16(tm + b * 64, make_desc64(hi, loF + 2 * k), make_desc64(hi, loWc + 2 * k), idesc64, k ? 1u : 0u);
        umma_commit(u_full + b);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_bf16(tm + b * 64 + 32, make_desc64(hi, loS + 2 * k), make_desc64(hi, loWcs + 2 * k), idesc, 1u);
        umma_commit(fs_empty + b);     // the operand stage may be refilled once these MMAs have read it
      }
      __syncwarp();
    }
  } else {
    // ================================ consumers: routing (U -> V tile) and Z -> shared memory ================================
    const int grp = warp >> 2, quad = warp & 3;
    const int m = quad * 32 + lane;                         // tile row = TMEM lane
    const uint32_t lane_addr = static_cast<uint32_t>(quad * 32) << 16;
    const float* zbv = reinterpret_cast<const float*>(tmem_slot + 4);   // zbias staged in shared memory by the prologue
    uint32_t it0 = 0, rn = 0;                               // tile counter at the start of the current (block, sample); pair counter
    for (int r = blockIdx.x; r < p.nregions; r += gridDim.x) {
      const int Y0 = (r / p.regions_x) * kHrRH - 1, X0 = (r % p.regions_x) * kHrRW - 1;
      for (int n = 0; n < p.batch; ++n, it0 += kHrTiles, ++rn) {
        __half* zdst = sZ + (rn & 1) * (kHrZK * kHrPix);
        for (int t = grp; t < kHrTiles; t += 2) {
          const uint32_t it = it0 + t;
          const int b = grp;                                // it & 1 == grp because it0 is a multiple of 4
          const uint32_t par = (it >> 1) & 1u;
          const int i = t * 128 + m;
          const int py = i / kHrPW, px = i - py * kHrPW;
          const int Y = Y0 + py, X = X0 + px;
          float4 rr = make_float4(0.f, 0.f, 0.f, 0.f);
          if (i < kHrPW * kHrPH && Y >= 0 && Y < p.H && X >= 0 && X < p.W)
            rr = __ldg(reinterpret_cast<const float4*>(p.table + (static_cast<long>(Y) * p.W + X) * 8 + 4));
          // ---- routing: U -> V
          mbar_wait(u_full + b, par);
          tc_fence_after();
          {
            uint32_t u0[16], u1[16];
            tmem_ld16(tm + lane_addr + b * 64, u0);
            tmem_ld16(tm + lane_addr + b * 64 + 16, u1);
            tmem_ld_wait();
            float tk[8];
#pragma unroll
            for (int k = 0; k < 8; ++k)
              tk[k] = rr.x * __uint_as_float(u0[k]) + rr.y * __uint_as_float(u0[8 + k]) + rr.z * __uint_as_float(u1[k]) + rr.w * __uint_as_float(u1[8 + k]);
            const float re[4] = {rr.x, rr.y, rr.z, rr.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              float v[8];
#pragma unroll
              for (int k = 0; k < 8; ++k) v[k] = re[e] * tk[k];
              *reinterpret_cast<uint4*>(sV + b * 16384 + swz(m, e)) = pack8(v, FMT);
            }
          }
          fence_proxy_async();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(v_full + b);
          // ---- Z (+ the fusion bias seen through the tail taps) -> shared memory as fp16 partial products
          mbar_wait(z_full + b, par);
          tc_fence_after();
          {
            uint32_t z0[16], z1[16];
            tmem_ld16(tm + lane_addr + b * 64 + 32, z0);
            tmem_ld16(tm + lane_addr + b * 64 + 48, z1);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(acc_empty + b);
            mbar_wait(zb_empty + (rn & 1), ((rn >> 1) & 1u) ^ 1u);      // the tail of pair rn - 2 has been summed
#pragma unroll
            for (int k = 0; k < 16; ++k) zdst[k * kHrPix + i] = __float2half_rn(__uint_as_float(z0[k]) + zbv[k]);
#pragma unroll
            for (int k = 16; k < kHrZK; ++k) zdst[k * kHrPix + i] = __float2half_rn(__uint_as_float(z1[k - 16]) + zbv[k]);
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(zb_full + (rn & 1));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kHrIssuerWarp) { tc_fence_after(); tmem_dealloc<128>(tm); }
}

}  // namespace savsr

using namespace savsr;

extern "C" int savsr_satu_index(savsr_ctx* ctx, const savsr_satu_weights* wts, int h, int w, int H, int W, float s_h,
                                float s_w, float* rel_y, float* rel_x, int32_t* cell_y, int32_t* cell_x, float* base_y,
                                float* base_x, int32_t* corner_y, int32_t* corner_x, float* table, savsr_stream st_) {
  SAVSR_REQUIRE(ctx, "savsr_satu_index: null context");
  DeviceGuard guard(ctx->device);
  SAVSR_REQUIRE(h >= 2 && w >= 2 && H >= 1 && W >= 1, "savsr_satu_index: bad sizes lr %dx%d hr %dx%d", h, w, H, W);
  SAVSR_REQUIRE(s_h > 0.f && s_w > 0.f, "savsr_satu_index: scale must be positive, got (%g, %g)", s_h, s_w);
  cudaStream_t st = static_cast<cudaStream_t>(st_);
  satu_axis_kernel<<<(H + 127) / 128, 128, 0, st>>>(H, h, s_h, rel_y, cell_y, base_y, corner_y);
  satu_axis_kernel<<<(W + 127) / 128, 128, 0, st>>>(W, w, s_w, rel_x, cell_x, base_x, corner_x);
  if (table) {
    SAVSR_REQUIRE(wts && wts->body0_w && wts->body0_b && wts->body2_w && wts->body2_b && wts->routing_w && wts->routing_b &&
                  wts->offset_w && wts->offset_b && wts->st_offset_w && wts->st_offset_b,
                  "savsr_satu_index: table requested but MLP weights missing");
    const long npix = static_cast<long>(H) * W;
    satu_table_kernel<<<static_cast<unsigned>((npix + 127) / 128), 128, 0, st>>>(*wts, H, W, s_h, s_w, table);
  }
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int savsr_satu_kconv_sta(savsr_ctx* ctx, savsr_arena* arena, int a_slot, int x_slot, int dst_slot, int h, int w,
                                    const void* weights, const float* bias, float slope, savsr_stream st) {
  SAVSR_REQUIRE(ctx && arena && weights && bias, "savsr_satu_kconv_sta: null pointer");
  SAVSR_REQUIRE(a_slot >= 0 && a_slot < arena->nslots && x_slot >= 0 && x_slot < arena->nslots && dst_slot >= 0 &&
                dst_slot < arena->nslots, "savsr_satu_kconv_sta: slot out of range");
  SAVSR_REQUIRE(dst_slot != a_slot && dst_slot != x_slot, "savsr_satu_kconv_sta: the destination slot must differ from both sources");
  SAVSR_REQUIRE(h >= 1 && w >= 1 && h <= arena->height && w <= arena->width, "savsr_satu_kconv_sta: region %dx%d exceeds arena", h, w);
  SAVSR_REQUIRE(slope >= 0.f && slope <= 1.f, "savsr_satu_kconv_sta: LeakyReLU slope %g outside [0, 1]", slope);
  if (arena->batch == 0) return 0;
  KstaParams p;
  memset(&p, 0, sizeof(p));
  p.tm_tile = arena->tm_tile;
  p.arena = arena->base;
  p.weights = static_cast<const uint8_t*>(weights);
  p.bias = bias;
  p.slope = slope;
  p.batch = arena->batch; p.hp = arena->height; p.wp = arena->width; p.h = h; p.w = w;
  p.a_slot = a_slot; p.x_slot = x_slot; p.dst_slot = dst_slot;
  p.tiles_x = arena->tiles_x; p.tiles_y = arena->tiles_y;
  const int tiles = p.tiles_x * p.tiles_y;
  p.nbatches = arena->batch * ((tiles + 1) / 2);
  p.chunk = (p.nbatches + ctx->sm_count - 1) / ctx->sm_count;
  p.fmt = ctx->fmt;
  const int grid = (p.nbatches + p.chunk - 1) / p.chunk;
  DeviceGuard guard(ctx->device);
  if (int rc = ensure_smem_attr(ctx, kAttrKsta, satu_kconv_sta_kernel, kKstaSmem)) return rc;
  satu_kconv_sta_kernel<<<grid, kKstaThreads, kKstaSmem, static_cast<cudaStream_t>(st)>>>(p);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

template <bool U8>
static int satu_hr(const char* name, savsr_ctx* ctx, savsr_arena* lr, int x_slot, int sta_slot, int h, int w, int H, int W, const float* table,
                   const float* base_y, const float* base_x, const void* weights, const float* zbias, const float* tail_bias,
                   const void* x_in, int t, int centre, void* out, savsr_stream st) {
  SAVSR_REQUIRE(ctx && lr && table && base_y && base_x && weights && zbias && tail_bias && x_in && out, "%s: null pointer", name);
  DeviceGuard guard(ctx->device);
  SAVSR_REQUIRE(x_slot >= 0 && x_slot < lr->nslots && sta_slot >= 0 && sta_slot < lr->nslots, "%s: LR slot out of range", name);
  SAVSR_REQUIRE(h >= 2 && w >= 2 && h <= lr->height && w <= lr->width, "%s: region %dx%d exceeds LR arena", name, h, w);
  SAVSR_REQUIRE(h < 65536 && w < 65536, "%s: LR frames larger than 65535 pixels per side are not supported", name);
  SAVSR_REQUIRE(H >= 1 && W >= 1 && t >= 1 && centre >= 0 && centre < t, "%s: bad HR size %dx%d or window (%d, %d)", name, H, W, t, centre);
  if (lr->batch == 0) return 0;
  const bool fp16 = ctx->fmt == SAVSR_FMT_FP16;
  auto kernel = fp16 ? satu_hr_kernel<SAVSR_FMT_FP16, U8> : satu_hr_kernel<SAVSR_FMT_BF16, U8>;
  const int bit = U8 ? kAttrSatuHrU8 + (fp16 ? 1 : 0) : (fp16 ? kAttrSatuHr : kAttrSatuHrBf16);
  if (int rc = ensure_smem_attr(ctx, bit, kernel, kHrSmem)) return rc;
  HrParams p;
  p.lr = lr->base; p.table = table; p.base_y = base_y; p.base_x = base_x;
  p.weights = static_cast<const uint8_t*>(weights); p.zbias = zbias; p.tail_bias = tail_bias; p.x_in = x_in; p.out = out;
  p.batch = lr->batch; p.hp = lr->height; p.wp = lr->width; p.h = h; p.w = w; p.H = H; p.W = W;
  p.x_slot = x_slot; p.sta_slot = sta_slot; p.t = t; p.centre = centre; p.fmt = ctx->fmt;
  p.regions_x = (W + kHrRW - 1) / kHrRW;
  p.nregions = p.regions_x * ((H + kHrRH - 1) / kHrRH);
  const int grid = p.nregions < ctx->sm_count ? p.nregions : ctx->sm_count;
  kernel<<<grid, kHrThreads, kHrSmem, static_cast<cudaStream_t>(st)>>>(p);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int savsr_satu_hr(savsr_ctx* ctx, savsr_arena* lr, int x_slot, int sta_slot, int h, int w, int H, int W,
                             const float* table, const float* base_y, const float* base_x, const void* weights,
                             const float* zbias, const float* tail_bias, const float* x_in, int t, int centre, float* out,
                             savsr_stream st) {
  return satu_hr<false>("savsr_satu_hr", ctx, lr, x_slot, sta_slot, h, w, H, W, table, base_y, base_x, weights, zbias, tail_bias, x_in, t,
                        centre, out, st);
}

extern "C" int savsr_satu_hr_u8(savsr_ctx* ctx, savsr_arena* lr, int x_slot, int sta_slot, int h, int w, int H, int W,
                                const float* table, const float* base_y, const float* base_x, const void* weights,
                                const float* zbias, const float* tail_bias, const uint8_t* x_in, int t, int centre, uint8_t* out,
                                savsr_stream st) {
  return satu_hr<true>("savsr_satu_hr_u8", ctx, lr, x_slot, sta_slot, h, w, H, W, table, base_y, base_x, weights, zbias, tail_bias, x_in, t,
                       centre, out, st);
}
