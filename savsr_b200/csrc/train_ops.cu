// Kernels of the native training step (row f1 of the scope table, stage B; lbasicsr/models/sr_model.py:101-128 runs the same
// step through autograd + cuDNN).  Everything here works on the SAME activation arena the forward kernels use (16-bit NHWC,
// C = 64) plus a second, pixel-contiguous arena ("T-arena": 16-bit NCHW with a padded row pitch) that feeds the weight-gradient
// contraction, whose K dimension is the pixel index:
//
//   savsr_slot_axpby          dst = alpha * x + beta * y on arena slots (residual adds, gradient accumulation)
//   savsr_grad_prep           g = (dV * cscale[n][c] + cadd[n][c]) * act'(out): the gradient entering a convolution, written back
//                             NHWC (operand of the data gradient), transposed NCHW (operand of the weight gradient), and summed
//                             into the bias gradient -- one pass over dV
//   savsr_slot_to_nchw3       an activation slot as three x-shifted NCHW copies (the other operand of the weight gradient)
//   savsr_pack_conv_chunks    table-driven weight packing: every filter of the net -> tensor-core blocks, forward orientation or
//                             transposed + flipped (data gradient), in ONE launch per step
//   savsr_conv_wgrad_batched  table-driven tcgen05 weight gradient: all (conv, source) pairs of a step in one persistent launch
//   savsr_adam_ema            Adam + EMA over the flat parameter / gradient / moment buffers
//   savsr_adam_ema_dev        the same with the learning rate read from device memory (a replayed graph follows a schedule)
#include "common.cuh"

namespace savsr {

constexpr int kMaxTrainEntries = 32;
// layouts the ctypes binding (savsr_b200/_capi.py) mirrors
static_assert(sizeof(savsr_axpby) == 20 && sizeof(savsr_nchw3) == 8 && sizeof(savsr_grad_prep_entry) == 72 && sizeof(savsr_pack_chunk) == 40 &&
              sizeof(savsr_wgrad_item) == 48, "C ABI struct layout changed: update savsr_b200/_capi.py and tests/test_boundary_cpu.py");

// ------------------------------------------------------------------------------------------------ slot axpby
struct AxpbyLaunch {
  uint16_t* arena;
  long slot_vecs;      // uint4 vectors per slot
  int n, fmt;
  savsr_axpby e[kMaxTrainEntries];
};

__device__ __forceinline__ uint32_t axpby_word(uint32_t a, uint32_t b, float alpha, float beta, int fmt) {
  return pack_h2(alpha * h_lo(a, fmt) + beta * h_lo(b, fmt), alpha * h_hi(a, fmt) + beta * h_hi(b, fmt), fmt);
}

__global__ void __launch_bounds__(256) slot_axpby_kernel(const __grid_constant__ AxpbyLaunch L) {
  pdl_wait();
  pdl_trigger();
  const savsr_axpby& e = L.e[blockIdx.y];
  const uint4* x = reinterpret_cast<const uint4*>(L.arena) + e.x_slot * L.slot_vecs;
  const uint4* y = e.y_slot >= 0 ? reinterpret_cast<const uint4*>(L.arena) + e.y_slot * L.slot_vecs : nullptr;
  uint4* d = reinterpret_cast<uint4*>(L.arena) + e.dst_slot * L.slot_vecs;
  const float alpha = e.alpha, beta = y ? e.beta : 0.f;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < L.slot_vecs; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const uint4 a = x[i];
    const uint4 b = y ? y[i] : make_uint4(0, 0, 0, 0);
    uint4 o;
    o.x = axpby_word(a.x, b.x, alpha, beta, L.fmt); o.y = axpby_word(a.y, b.y, alpha, beta, L.fmt);
    o.z = axpby_word(a.z, b.z, alpha, beta, L.fmt); o.w = axpby_word(a.w, b.w, alpha, beta, L.fmt);
    d[i] = o;
  }
}

// ------------------------------------------------------------------------------------------------ NHWC -> NCHW transposers
// One block = one image row of one entry.  A 64-pixel chunk of the row sits in shared memory as [pixel][33 words] (64 channels
// + one pad word: conflict-free 32-bit writes, at most 2-way conflicts on the transposed 16-bit reads); it is written out as
// 16-byte vectors of 8 consecutive pixels of one channel plane, 8 lanes covering one 128-byte line.
struct GradPrepLaunch {
  uint16_t* arena;
  uint16_t* tbase;
  int batch, height, width, pitch, n, fmt;
  savsr_grad_prep_entry e[kMaxTrainEntries];
};

// tile word address of (pixel row r, channel-pair word w): 33 words per row, and rows >= 32 shifted by 4 banks so that the eight
// 8-pixel segments a warp reads in the transposed pass fall into distinct banks
__device__ __forceinline__ int tile_word(int r, int w) { return r * 33 + (r >> 5) * 4 + w; }
constexpr int kTileWords = 66 * 33 + 12;

// One thread = one channel PAIR x 8 consecutive pixels: eight 32-bit shared loads -> two 16-byte global stores (channels 2cp, 2cp+1).
__device__ __forceinline__ void store_plane_pair(uint16_t* plane_row0, long plane_elems, const uint32_t* tile, int seg, int cp, int row_shift) {
  uint32_t w[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) w[j] = tile[tile_word(seg * 8 + j + row_shift, cp)];
  uint4 lo, hi;
  lo.x = (w[0] & 0xffffu) | (w[1] << 16); hi.x = (w[0] >> 16) | (w[1] & 0xffff0000u);
  lo.y = (w[2] & 0xffffu) | (w[3] << 16); hi.y = (w[2] >> 16) | (w[3] & 0xffff0000u);
  lo.z = (w[4] & 0xffffu) | (w[5] << 16); hi.z = (w[4] >> 16) | (w[5] & 0xffff0000u);
  lo.w = (w[6] & 0xffffu) | (w[7] << 16); hi.w = (w[6] >> 16) | (w[7] & 0xffff0000u);
  *reinterpret_cast<uint4*>(plane_row0 + (2 * cp) * plane_elems + seg * 8) = lo;
  *reinterpret_cast<uint4*>(plane_row0 + (2 * cp + 1) * plane_elems + seg * 8) = hi;
}

__global__ void __launch_bounds__(256) grad_prep_kernel(const __grid_constant__ GradPrepLaunch L) {
  __shared__ uint32_t tile[kTileWords];
  pdl_wait();
  pdl_trigger();
  const savsr_grad_prep_entry& e = L.e[blockIdx.z];
  const int y = blockIdx.x, n = blockIdx.y, t = threadIdx.x, fmt = L.fmt;
  const long row_elems = static_cast<long>(L.width) * kC;
  const long slot_elems = static_cast<long>(L.batch) * L.height * row_elems;
  const long row_off = (static_cast<long>(n) * L.height + y) * row_elems;
  const uint16_t* dv = L.arena + e.dv_slot * slot_elems + row_off;
  const uint16_t* ao = e.act != SAVSR_ACT_NONE ? L.arena + e.out_slot * slot_elems + row_off : nullptr;
  uint16_t* gd = e.g_slot >= 0 ? L.arena + e.g_slot * slot_elems + row_off : nullptr;
  const int ch8 = t & 7;
  float cs[8], ca[8], db[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    cs[j] = e.cscale ? __ldg(e.cscale + static_cast<long>(n) * e.cscale_stride + ch8 * 8 + j) : 1.f;
    ca[j] = e.cadd ? e.cadd_mul * __ldg(e.cadd + static_cast<long>(n) * e.cadd_stride + ch8 * 8 + j) : 0.f;
    db[j] = 0.f;
  }
  const float neg = e.act == SAVSR_ACT_LRELU ? e.slope : 0.f;
  const long plane_elems = static_cast<long>(L.height) * L.pitch;
  uint16_t* tplane = e.gt_tslot >= 0 ? L.tbase + ((static_cast<long>(e.gt_tslot) * L.batch + n) * kC) * plane_elems + static_cast<long>(y) * L.pitch : nullptr;
  for (int x0 = 0; x0 < L.width; x0 += 64) {
    __syncthreads();
    for (int pp = t >> 3; pp < 64; pp += 32) {
      const int x = x0 + pp;
      uint4 o = make_uint4(0, 0, 0, 0);
      if (x < L.width) {
        const uint4 d = *reinterpret_cast<const uint4*>(dv + x * kC + ch8 * 8);
        uint4 a = make_uint4(0, 0, 0, 0);
        if (ao) a = *reinterpret_cast<const uint4*>(ao + x * kC + ch8 * 8);
        const uint32_t dw[4] = {d.x, d.y, d.z, d.w}, aw[4] = {a.x, a.y, a.z, a.w};
        uint32_t ow[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float g0 = h_lo(dw[j], fmt) * cs[2 * j] + ca[2 * j], g1 = h_hi(dw[j], fmt) * cs[2 * j + 1] + ca[2 * j + 1];
          if (ao) {
            if (!(h_lo(aw[j], fmt) > 0.f)) g0 *= neg;
            if (!(h_hi(aw[j], fmt) > 0.f)) g1 *= neg;
          }
          ow[j] = pack_h2(g0, g1, fmt);
          db[2 * j] += h_lo(ow[j], fmt); db[2 * j + 1] += h_hi(ow[j], fmt);     // the bias gradient sums what the weight gradient sees
        }
        o = make_uint4(ow[0], ow[1], ow[2], ow[3]);
        if (gd) *reinterpret_cast<uint4*>(gd + x * kC + ch8 * 8) = o;
      }
      uint32_t* tw = tile + tile_word(pp, ch8 * 4);
      tw[0] = o.x; tw[1] = o.y; tw[2] = o.z; tw[3] = o.w;
    }
    __syncthreads();
    if (tplane) {
      const int seg = t & 7, cp = t >> 3;
      if (x0 + seg * 8 < L.pitch) store_plane_pair(tplane + x0, plane_elems, tile, seg, cp, 0);
    }
  }
  if (e.dbias) {
    // lanes l, l+8, l+16, l+24 of a warp hold the same eight channels: two shuffle steps, then one row of partials per warp
    // (shared-memory float atomics compile to CAS loops: measured as the top stall of the first version of this kernel)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      db[j] += __shfl_xor_sync(0xffffffffu, db[j], 8);
      db[j] += __shfl_xor_sync(0xffffffffu, db[j], 16);
    }
    __syncthreads();                                   // the tile is free: reuse it as [8 warps][64 channels]
    float* part = reinterpret_cast<float*>(tile);
    if ((t & 31) < 8) {
#pragma unroll
      for (int j = 0; j < 8; ++j) part[(t >> 5) * 64 + ch8 * 8 + j] = db[j];
    }
    __syncthreads();
    if (t < 64) {
      float v = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) v += part[w * 64 + t];
      atomicAdd(e.dbias + t, v);
    }
  }
}

struct Nchw3Launch {
  const uint16_t* arena;
  uint16_t* tbase;
  int batch, height, width, pitch, n;
  savsr_nchw3 e[kMaxTrainEntries];
};

// copy d (d = 0, 1, 2) holds X[.., x + d - 1], zero where that leaves the row: the tile carries one halo pixel on each side
__global__ void __launch_bounds__(256) slot_to_nchw3_kernel(const __grid_constant__ Nchw3Launch L) {
  __shared__ uint32_t tile[kTileWords];
  const savsr_nchw3& e = L.e[blockIdx.z];
  const int y = blockIdx.x, n = blockIdx.y, t = threadIdx.x;
  const long row_elems = static_cast<long>(L.width) * kC;
  const long slot_elems = static_cast<long>(L.batch) * L.height * row_elems;
  const uint16_t* src = L.arena + e.x_slot * slot_elems + (static_cast<long>(n) * L.height + y) * row_elems;
  const long plane_elems = static_cast<long>(L.height) * L.pitch;
  const long tslot_elems = static_cast<long>(L.batch) * kC * plane_elems;
  uint16_t* tplane = L.tbase + static_cast<long>(e.t_slot) * tslot_elems + (static_cast<long>(n) * kC) * plane_elems + static_cast<long>(y) * L.pitch;
  for (int x0 = 0; x0 < L.width; x0 += 64) {
    __syncthreads();
    for (int idx = t; idx < 66 * 8; idx += 256) {
      const int pp = idx >> 3, ch8 = idx & 7, x = x0 - 1 + pp;
      uint4 o = make_uint4(0, 0, 0, 0);
      if (x >= 0 && x < L.width) o = *reinterpret_cast<const uint4*>(src + x * kC + ch8 * 8);
      uint32_t* tw = tile + tile_word(pp, ch8 * 4);
      tw[0] = o.x; tw[1] = o.y; tw[2] = o.z; tw[3] = o.w;
    }
    __syncthreads();
    const int seg = t & 7, cp = t >> 3;
#pragma unroll
    for (int d = 0; d < 3; ++d)
      if (x0 + seg * 8 < L.pitch) store_plane_pair(tplane + d * tslot_elems + x0, plane_elems, tile, seg, cp, d);
  }
}

// ------------------------------------------------------------------------------------------------ table-driven weight packing
// One block per chunk = the k*k [64][64] tensor-core blocks of one (64 output channels, 64 input channels) corner of a filter,
// rows in SAVSR_ROWS_QUAD order, 128-byte swizzle.  transposed: the data-gradient operand (rows = input channels, K = output
// channels, taps flipped).
__global__ void __launch_bounds__(256) pack_chunks_kernel(const savsr_pack_chunk* __restrict__ chunks, int fmt) {
  const savsr_pack_chunk ch = chunks[blockIdx.x];
  const int taps = ch.ksize * ch.ksize;
  uint16_t* out = static_cast<uint16_t*>(ch.dst);
  for (int idx = threadIdx.x; idx < taps * 4096; idx += blockDim.x) {
    const int k = idx & 63, n = (idx >> 6) & 63, tap = idx >> 12;
    const int r = quad_row(n);
    float val;
    if (ch.transposed) {
      const int o = ch.o_base + k, i = ch.i_base + r;
      val = (o < ch.co_total && i < ch.ci_total) ? __ldg(ch.w + (static_cast<long>(o) * ch.ci_total + i) * taps + (taps - 1 - tap)) : 0.f;
    } else {
      const int o = ch.o_base + r, i = ch.i_base + k;
      val = (o < ch.co_total && i < ch.ci_total) ? __ldg(ch.w + (static_cast<long>(o) * ch.ci_total + i) * taps + tap) : 0.f;
    }
    out[tap * 4096 + n * 64 + ((((k >> 3) ^ (n & 7)) << 3) | (k & 7))] = float_to_h(val, fmt);
  }
}

// ------------------------------------------------------------------------------------------------ batched weight gradient
// The kernel of conv_wgrad.cu with its problem description read from a device table: item = one (convolution, 64-channel
// source) pair; work unit = (item, sample, 64-pixel x segment, row chunk).  A = two stacked x-shifted X tiles (M = 128),
// B = the dY tile (N = 64), six 64-column accumulators in TMEM, flushed with fp32 atomics whenever the weight block changes.
struct WgradBatchedParams {
  CUtensorMap tm;        // the whole T-arena as [planes][H][pitch], box (64 px, 1 row, 64 planes)
  const savsr_wgrad_item* items;
  int batch, height, width;
  int nxseg, nychunk, rows_per_chunk;
  int nunits, chunk;
  int fmt;
};

constexpr int kWbRowSlots = 4;
constexpr int kWbRowBytes = 4 * 8192;
constexpr int kWbDyStages = 2;
constexpr int kWbThreads = 6 * 32;
constexpr int kWbSmem = 1024 + kWbRowSlots * kWbRowBytes + kWbDyStages * 8192 + 256;

__device__ __forceinline__ void tma_load_3d_t(void* smem_dst, const CUtensorMap* tm, uint64_t* bar, int x, int y, int c) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(x), "r"(y), "r"(c), "r"(smem_u32(bar))
      : "memory");
}

struct WbUnit { int item, n, x0, y0, y1; };
__device__ __forceinline__ WbUnit wb_unit(const WgradBatchedParams& p, int u) {
  WbUnit it;
  const int yc = u % p.nychunk; u /= p.nychunk;
  const int xs = u % p.nxseg; u /= p.nxseg;
  it.n = u % p.batch;
  it.item = u / p.batch;
  it.x0 = xs * 64;
  it.y0 = yc * p.rows_per_chunk;
  it.y1 = min(it.y0 + p.rows_per_chunk, p.height);
  return it;
}

__global__ void __launch_bounds__(kWbThreads, 1) conv_wgrad_batched_kernel(const __grid_constant__ WgradBatchedParams p) {
  extern __shared__ uint8_t raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* s_rows = smem;
  uint8_t* s_dy = smem + kWbRowSlots * kWbRowBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_dy + kWbDyStages * 8192);
  uint64_t* row_full = bars;
  uint64_t* row_empty = bars + 4;
  uint64_t* dy_full = bars + 8;
  uint64_t* dy_empty = bars + 10;
  uint64_t* acc_full = bars + 12;
  uint64_t* acc_empty = bars + 13;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 14);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int u_begin = blockIdx.x * p.chunk, u_end = min(u_begin + p.chunk, p.nunits);
  if (threadIdx.x == 0) {
    prefetch_tensormap(&p.tm);
    for (int i = 0; i < 4; ++i) { mbar_init(row_full + i, 1); mbar_init(row_empty + i, 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(dy_full + i, 1); mbar_init(dy_empty + i, 1); }
    mbar_init(acc_full, 1); mbar_init(acc_empty, 4);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tm = *tmem_slot;
  const int planes_per_tslot = p.batch * kC;

  if (warp == 0) {
    // ================================ TMA producer ================================
    if (lane == 0) {
      uint32_t rcount = 0, dcount = 0;
      for (int u = u_begin; u < u_end; ++u) {
        const WbUnit w = wb_unit(p, u);
        const int xt = __ldg(&p.items[w.item].x_tslot), gt = __ldg(&p.items[w.item].g_tslot);
        const int cx = xt * planes_per_tslot + w.n * kC, cy = gt * planes_per_tslot + w.n * kC;
        for (int r = w.y0 - 1; r <= w.y1; ++r, ++rcount) {
          const int slot = rcount & 3;
          mbar_wait(row_empty + slot, ((rcount >> 2) & 1u) ^ 1u);
          mbar_expect_tx(row_full + slot, 3 * 8192u);
#pragma unroll
          for (int dx = 0; dx < 3; ++dx)
            tma_load_3d_t(s_rows + slot * kWbRowBytes + dx * 8192, &p.tm, row_full + slot, w.x0, r, dx * planes_per_tslot + cx);   // rows outside the image read as zero
          const int y = r - 1;
          if (y >= w.y0) {
            const int st = dcount & 1;
            mbar_wait(dy_empty + st, ((dcount >> 1) & 1u) ^ 1u);
            mbar_expect_tx(dy_full + st, 8192u);
            tma_load_3d_t(s_dy + st * 8192, &p.tm, dy_full + st, w.x0, y, cy);
            ++dcount;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ================================
    const uint32_t idesc = umma_idesc_f16(64, p.fmt);
    constexpr uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);
    const uint32_t lo_rows = (smem_u32(s_rows) >> 4) & 0x3fffu, lo_dy = (smem_u32(s_dy) >> 4) & 0x3fffu;
    uint32_t rcount = 0, dcount = 0, flushes = 0;
    int cur_key = -1;
    bool fresh = true;
    for (int u = u_begin; u < u_end; ++u) {
      const WbUnit w = wb_unit(p, u);
      const int key = w.item * p.batch + (__ldg(&p.items[w.item].per_sample) ? w.n : 0);
      if (key != cur_key && cur_key >= 0) {
        if (elect_one()) umma_commit(acc_full);
        __syncwarp();
        mbar_wait(acc_empty, flushes & 1u);
        ++flushes;
        tc_fence_after();
        fresh = true;
      }
      cur_key = key;
      for (int y = w.y0; y < w.y1; ++y) {
        const uint32_t base = rcount + (y - w.y0);
        if (y == w.y0) {
          mbar_wait(row_full + (base & 3), (base >> 2) & 1u);
          mbar_wait(row_full + ((base + 1) & 3), ((base + 1) >> 2) & 1u);
        }
        mbar_wait(row_full + ((base + 2) & 3), ((base + 2) >> 2) & 1u);
        const int st = dcount & 1;
        mbar_wait(dy_full + st, (dcount >> 1) & 1u);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t bl = lo_dy + st * (8192 >> 4);
#pragma unroll
          for (int dy = 0; dy < 3; ++dy) {
            const uint32_t al = lo_rows + ((base + dy) & 3) * (kWbRowBytes >> 4);
#pragma unroll
            for (int pair = 0; pair < 2; ++pair) {
              const uint32_t d = tm + static_cast<uint32_t>((dy * 2 + pair) * 64);
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma_bf16(d, (static_cast<uint64_t>(hi) << 32) | (al + pair * (16384 >> 4) + 2 * k), (static_cast<uint64_t>(hi) << 32) | (bl + 2 * k), idesc,
                          (fresh && k == 0) ? 0u : 1u);
            }
          }
          umma_commit(dy_empty + st);
          umma_commit(row_empty + (base & 3));
          if (y == w.y1 - 1) {
            umma_commit(row_empty + ((base + 1) & 3));
            umma_commit(row_empty + ((base + 2) & 3));
          }
        }
        __syncwarp();
        fresh = false;
        ++dcount;
      }
      rcount += static_cast<uint32_t>(w.y1 - w.y0 + 2);
    }
    if (cur_key >= 0) {
      if (elect_one()) umma_commit(acc_full);
      __syncwarp();
    }
  } else {
    // ================================ flush warps ================================
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    int cur_key = -1, cur_item = 0, cur_n = 0;
    uint32_t flushes = 0;
    auto flush = [&]() {
      mbar_wait(acc_full, flushes & 1u);
      ++flushes;
      tc_fence_after();
      const savsr_wgrad_item it = p.items[cur_item];
      float* dwb = it.dw + (it.per_sample ? static_cast<long>(cur_n) * it.sample_stride : 0);
      const int i = it.ci_off + (row & 63);
      const int taps = it.ksize == 1 ? 1 : 9;
#pragma unroll 1
      for (int acc = 0; acc < 6; ++acc) {
        const int dy = acc >> 1, pair = acc & 1;
        const int dx = pair == 0 ? (row < 64 ? 0 : 1) : (row < 64 ? 2 : -1);
        const bool want = dx >= 0 && (taps == 9 || (dy == 1 && dx == 1));     // a 1x1 filter takes the centre tap only
        const int tap = taps == 9 ? dy * 3 + dx : 0;
        uint32_t v[16];
#pragma unroll 1
        for (int c0 = 0; c0 < 64; c0 += 16) {
          tmem_ld16(tm + (static_cast<uint32_t>(quad * 32) << 16) + static_cast<uint32_t>(acc * 64 + c0), v);
          tmem_ld_wait();
          if (want) {
            if (it.layout == SAVSR_WGRAD_TIO) {
              // [tap][input channel][64 output channels]: this thread's 16 accumulator columns are contiguous -> four 16-byte reductions
              float4* dst = reinterpret_cast<float4*>(dwb + (static_cast<long>(tap) * it.ci_total + i) * 64 + it.o_off + c0);
#pragma unroll
              for (int q = 0; q < 4; ++q)
                atomicAdd(dst + q, make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3])));
            } else {
#pragma unroll
              for (int c = 0; c < 16; ++c)
                atomicAdd(dwb + (static_cast<long>(it.o_off + c0 + c) * it.ci_total + i) * taps + tap, __uint_as_float(v[c]));
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty);
    };
    for (int u = u_begin; u < u_end; ++u) {
      const WbUnit w = wb_unit(p, u);
      const int key = w.item * p.batch + (__ldg(&p.items[w.item].per_sample) ? w.n : 0);
      if (key != cur_key && cur_key >= 0) flush();
      cur_key = key; cur_item = w.item; cur_n = w.n;
    }
    if (cur_key >= 0) flush();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) { tc_fence_after(); tmem_dealloc<512>(tm); }
}

typedef CUresult (*EncodeTiledFnT)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// ------------------------------------------------------------------------------------------------ Adam + EMA
__global__ void __launch_bounds__(256) adam_ema_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                       float* __restrict__ v, float* __restrict__ ema, long n, float lr,
                                                       const float* __restrict__ lr_dev, float b1, float b2, float eps,
                                                       const float* __restrict__ step, float decay, float gscale) {
  const float t = *step;
  const float lr_t = lr_dev ? *lr_dev : lr;          // device-resident lr: a replayed CUDA graph follows a schedule
  const float bc1 = 1.f - powf(b1, t), bc2s = sqrtf(1.f - powf(b2, t));
  const float step_size = lr_t / bc1;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const float gi = g[i] * gscale;
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    const float pi = p[i] - step_size * (mi / (sqrtf(vi) / bc2s + eps));
    p[i] = pi;
    if (ema) ema[i] = decay * ema[i] + (1.f - decay) * pi;
  }
}

}  // namespace savsr

using namespace savsr;

extern "C" int savsr_slot_axpby(savsr_ctx* ctx, savsr_arena* arena, const savsr_axpby* entries, int n, savsr_stream st) {
  SAVSR_REQUIRE(ctx && arena && entries, "savsr_slot_axpby: null pointer");
  SAVSR_REQUIRE(n >= 0 && n <= kMaxTrainEntries, "savsr_slot_axpby: %d entries, at most %d per launch", n, kMaxTrainEntries);
  if (n == 0) return 0;
  DeviceGuard guard(ctx->device);
  AxpbyLaunch L;
  L.arena = reinterpret_cast<uint16_t*>(arena->base);
  L.slot_vecs = static_cast<long>(arena->batch) * arena->height * arena->width * kC / 8;
  L.n = n; L.fmt = ctx->fmt;
  for (int i = 0; i < n; ++i) {
    const savsr_axpby& e = entries[i];
    SAVSR_REQUIRE(e.dst_slot >= 0 && e.dst_slot < arena->nslots && e.x_slot >= 0 && e.x_slot < arena->nslots && e.y_slot < arena->nslots,
                  "savsr_slot_axpby: entry %d has a slot out of range", i);
    L.e[i] = e;
  }
  long blocks = (L.slot_vecs + 255) / 256;
  if (blocks > 4 * ctx->sm_count) blocks = 4 * ctx->sm_count;
  SAVSR_CUDA(launch_k(ctx->opt[SAVSR_OPT_PDL] != 0, slot_axpby_kernel, dim3(static_cast<unsigned>(blocks), n), dim3(256), 0, static_cast<cudaStream_t>(st), L));
  return 0;
}

static int check_tarena(const char* who, const savsr_arena* arena, const void* tbase, int pitch) {
  SAVSR_REQUIRE(tbase && (reinterpret_cast<uintptr_t>(tbase) & 15) == 0, "%s: the T-arena must be a 16-byte aligned device pointer", who);
  SAVSR_REQUIRE(pitch >= arena->width && pitch % 8 == 0, "%s: row pitch %d must be >= width %d and a multiple of 8 elements", who, pitch, arena->width);
  return 0;
}

extern "C" int savsr_grad_prep(savsr_ctx* ctx, savsr_arena* arena, void* tbase, int ntslots, int pitch, const savsr_grad_prep_entry* entries,
                               int n, savsr_stream st) {
  SAVSR_REQUIRE(ctx && arena && entries, "savsr_grad_prep: null pointer");
  SAVSR_REQUIRE(n >= 0 && n <= kMaxTrainEntries, "savsr_grad_prep: %d entries, at most %d per launch", n, kMaxTrainEntries);
  if (n == 0) return 0;
  DeviceGuard guard(ctx->device);
  GradPrepLaunch L;
  L.arena = reinterpret_cast<uint16_t*>(arena->base);
  L.tbase = static_cast<uint16_t*>(tbase);
  L.batch = arena->batch; L.height = arena->height; L.width = arena->width; L.pitch = pitch; L.n = n; L.fmt = ctx->fmt;
  bool any_t = false;
  for (int i = 0; i < n; ++i) {
    const savsr_grad_prep_entry& e = entries[i];
    SAVSR_REQUIRE(e.dv_slot >= 0 && e.dv_slot < arena->nslots && e.g_slot < arena->nslots, "savsr_grad_prep: entry %d has a slot out of range", i);
    SAVSR_REQUIRE(e.act == SAVSR_ACT_NONE || (e.out_slot >= 0 && e.out_slot < arena->nslots), "savsr_grad_prep: entry %d needs the stored output for its activation", i);
    SAVSR_REQUIRE(e.gt_tslot < ntslots, "savsr_grad_prep: entry %d T-slot %d out of range [0,%d)", i, e.gt_tslot, ntslots);
    any_t |= e.gt_tslot >= 0;
    L.e[i] = e;
  }
  if (any_t) if (int rc = check_tarena("savsr_grad_prep", arena, tbase, pitch)) return rc;
  SAVSR_CUDA(launch_k(ctx->opt[SAVSR_OPT_PDL] != 0, grad_prep_kernel, dim3(arena->height, arena->batch, n), dim3(256), 0, static_cast<cudaStream_t>(st), L));
  return 0;
}

extern "C" int savsr_slot_to_nchw3(savsr_ctx* ctx, savsr_arena* arena, void* tbase, int ntslots, int pitch, const savsr_nchw3* entries, int n,
                                   savsr_stream st) {
  SAVSR_REQUIRE(ctx && arena && entries, "savsr_slot_to_nchw3: null pointer");
  SAVSR_REQUIRE(n >= 0 && n <= kMaxTrainEntries, "savsr_slot_to_nchw3: %d entries, at most %d per launch", n, kMaxTrainEntries);
  if (n == 0) return 0;
  DeviceGuard guard(ctx->device);
  if (int rc = check_tarena("savsr_slot_to_nchw3", arena, tbase, pitch)) return rc;
  Nchw3Launch L;
  L.arena = reinterpret_cast<const uint16_t*>(arena->base);
  L.tbase = static_cast<uint16_t*>(tbase);
  L.batch = arena->batch; L.height = arena->height; L.width = arena->width; L.pitch = pitch; L.n = n;
  for (int i = 0; i < n; ++i) {
    const savsr_nchw3& e = entries[i];
    SAVSR_REQUIRE(e.x_slot >= 0 && e.x_slot < arena->nslots, "savsr_slot_to_nchw3: entry %d slot out of range", i);
    SAVSR_REQUIRE(e.t_slot >= 0 && e.t_slot + 3 <= ntslots, "savsr_slot_to_nchw3: entry %d T-slots [%d, %d) out of range [0,%d)", i, e.t_slot, e.t_slot + 3, ntslots);
    L.e[i] = e;
  }
  slot_to_nchw3_kernel<<<dim3(arena->height, arena->batch, n), 256, 0, static_cast<cudaStream_t>(st)>>>(L);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int savsr_pack_conv_chunks(savsr_ctx* ctx, const savsr_pack_chunk* chunks_dev, int first, int count, savsr_stream st) {
  SAVSR_REQUIRE(ctx && chunks_dev, "savsr_pack_conv_chunks: null pointer");
  SAVSR_REQUIRE(first >= 0 && count >= 0, "savsr_pack_conv_chunks: bad range [%d, +%d)", first, count);
  if (count == 0) return 0;
  DeviceGuard guard(ctx->device);
  pack_chunks_kernel<<<count, 256, 0, static_cast<cudaStream_t>(st)>>>(chunks_dev + first, ctx->fmt);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int savsr_conv_wgrad_batched(savsr_ctx* ctx, const void* tbase, int ntslots, int batch, int height, int width, int pitch,
                                        const savsr_wgrad_item* items_dev, int first, int count, savsr_stream st) {
  SAVSR_REQUIRE(ctx && tbase && items_dev, "savsr_conv_wgrad_batched: null pointer");
  SAVSR_REQUIRE(batch >= 1 && height >= 1 && width >= 1 && ntslots >= 1, "savsr_conv_wgrad_batched: empty problem");
  SAVSR_REQUIRE(pitch >= width && pitch % 8 == 0, "savsr_conv_wgrad_batched: row pitch %d must be >= width %d and a multiple of 8 elements", pitch, width);
  SAVSR_REQUIRE((reinterpret_cast<uintptr_t>(tbase) & 15) == 0, "savsr_conv_wgrad_batched: the T-arena must be 16-byte aligned");
  SAVSR_REQUIRE(first >= 0 && count >= 0, "savsr_conv_wgrad_batched: bad range [%d, +%d)", first, count);
  if (count == 0) return 0;
  DeviceGuard guard(ctx->device);
  WgradBatchedParams p;
  memset(&p, 0, sizeof(p));
  {
    const long planes = static_cast<long>(ntslots) * batch * kC;
    const cuuint64_t dims[3] = {static_cast<cuuint64_t>(pitch), static_cast<cuuint64_t>(height), static_cast<cuuint64_t>(planes)};
    const cuuint64_t strides[2] = {static_cast<cuuint64_t>(pitch) * 2, static_cast<cuuint64_t>(pitch) * height * 2};
    const cuuint32_t box[3] = {64, 1, 64};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = reinterpret_cast<EncodeTiledFnT>(ctx->encode_tiled)(
        &p.tm, CU_TENSOR_MAP_DATA_TYPE_UINT16, 3, const_cast<void*>(tbase), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    SAVSR_REQUIRE(r == CUDA_SUCCESS, "savsr_conv_wgrad_batched: cuTensorMapEncodeTiled failed with CUresult %d (planes %ld, %dx%d)",
                  static_cast<int>(r), planes, height, pitch);
  }
  p.items = items_dev + first;
  p.batch = batch; p.height = height; p.width = width;
  p.nxseg = (width + 63) / 64;
  const long base_units = static_cast<long>(count) * batch * p.nxseg;
  long chunks = (2L * ctx->sm_count + base_units - 1) / base_units;       // about two units per SM when the table is short
  if (chunks > height) chunks = height;
  if (chunks < 1) chunks = 1;
  p.rows_per_chunk = static_cast<int>((height + chunks - 1) / chunks);
  p.nychunk = (height + p.rows_per_chunk - 1) / p.rows_per_chunk;
  const long nunits = base_units * p.nychunk;
  SAVSR_REQUIRE(nunits < (1L << 30), "savsr_conv_wgrad_batched: too many work units (%ld)", nunits);
  p.nunits = static_cast<int>(nunits);
  p.chunk = (p.nunits + ctx->sm_count - 1) / ctx->sm_count;
  p.fmt = ctx->fmt;
  const int grid = (p.nunits + p.chunk - 1) / p.chunk;
  if (int rc = ensure_smem_attr(ctx, kAttrWgradBatched, conv_wgrad_batched_kernel, kWbSmem)) return rc;
  conv_wgrad_batched_kernel<<<grid, kWbThreads, kWbSmem, static_cast<cudaStream_t>(st)>>>(p);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

static int launch_adam_ema(const char* who, savsr_ctx* ctx, float* param, const float* grad, float* exp_avg, float* exp_avg_sq, float* ema, long n,
                           float lr, const float* lr_dev, float beta1, float beta2, float eps, const float* step_dev, float ema_decay,
                           float grad_scale, savsr_stream st) {
  SAVSR_REQUIRE(ctx && param && grad && exp_avg && exp_avg_sq && step_dev, "%s: null pointer", who);
  SAVSR_REQUIRE(n >= 0, "%s: negative length", who);
  if (n == 0) return 0;
  DeviceGuard guard(ctx->device);
  long blocks = (n + 255) / 256;
  if (blocks > 8L * ctx->sm_count) blocks = 8L * ctx->sm_count;
  adam_ema_kernel<<<static_cast<unsigned>(blocks), 256, 0, static_cast<cudaStream_t>(st)>>>(param, grad, exp_avg, exp_avg_sq, ema, n, lr, lr_dev, beta1,
                                                                                          beta2, eps, step_dev, ema_decay, grad_scale);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int savsr_adam_ema(savsr_ctx* ctx, float* param, const float* grad, float* exp_avg, float* exp_avg_sq, float* ema, long n, float lr,
                              float beta1, float beta2, float eps, const float* step_dev, float ema_decay, float grad_scale, savsr_stream st) {
  return launch_adam_ema("savsr_adam_ema", ctx, param, grad, exp_avg, exp_avg_sq, ema, n, lr, nullptr, beta1, beta2, eps, step_dev, ema_decay,
                         grad_scale, st);
}

extern "C" int savsr_adam_ema_dev(savsr_ctx* ctx, float* param, const float* grad, float* exp_avg, float* exp_avg_sq, float* ema, long n,
                                  const float* lr_dev, float beta1, float beta2, float eps, const float* step_dev, float ema_decay, float grad_scale,
                                  savsr_stream st) {
  SAVSR_REQUIRE(lr_dev, "savsr_adam_ema_dev: null lr pointer");
  return launch_adam_ema("savsr_adam_ema_dev", ctx, param, grad, exp_avg, exp_avg_sq, ema, n, 0.f, lr_dev, beta1, beta2, eps, step_dev, ema_decay,
                         grad_scale, st);
}
