// Train-mode attention paths of the native training step (row f1, stage B): the scale-attention prologue of OSA-Conv with
// batch-statistics BatchNorm and its backward (savsr_arch.py:91-96, 123-128, 139-172), and the backward of the RCAB channel
// attention (savsr_arch.py:514-524).  Small problems (a batch of B <= 32 vectors of <= 640 elements, weight banks of a few MB):
// latency-bound CUDA-core kernels whose job is to replace ~100 framework launches per convolution by 3-4.
//
// Forward:   savsr_osa_prologue's pooling and routing kernels (small_ops.cu), then osa_assemble_train_kernel: z = ReLU(BN_batch(fc v)),
//            the four heads, and the per-sample folded kernel written TWICE: forward operand and transposed + flipped operand
//            (data gradient), both in the tensor-core block layout.
// Backward:  osa_unfold_bwd_kernel   dWfold -> d bank, d ca / fa / sa / ka            (thread = one (o, i) filter position)
//            osa_attn_chain_kernel   heads -> BatchNorm -> fc -> scale_routing, vectors only (one CTA per convolution)
//            osa_attn_wgrad_kernel   every weight / bias gradient of those layers as batch-summed outer products
#include "common.cuh"

namespace savsr {

constexpr int kMaxOsaT = 4;
static_assert(sizeof(savsr_osa_train) == 56 && sizeof(savsr_osa_grads) == 160, "C ABI struct layout changed: update savsr_b200/_capi.py");
// Samples per launch of the train-mode attention kernels.  Their per-sample arrays live in dynamic shared memory sized by the batch;
// the chain kernel needs the most (178 KB at 32 samples and ci = 320) and would pass the 227 KB a block may use at 42.
constexpr int kMaxBatchT = 32;
__host__ __device__ inline int osat_scratch_stride(int ci) { return 5 * ci + 192; }
__host__ __device__ inline int osat_off_h1(int ci) { return ci + 8; }
__host__ __device__ inline int osat_off_v2(int ci) { return 3 * ci + 8; }
__host__ __device__ inline int osat_off_att(int ci) { return 4 * ci + 8; }
__device__ __forceinline__ float sigmoid_t(float x) { return 1.f / (1.f + expf(-x)); }

struct OsaTrainLaunch {
  savsr_osa_params c[kMaxOsaT];
  savsr_osa_train t[kMaxOsaT];
  savsr_osa_grads g[kMaxOsaT];
  int nconvs, batch, fmt;
};

// state layout per conv: zpre [B][32] | z [B][32] | mu [32] | rstd [32]
__host__ __device__ inline int st_zpre(int b) { return b * 32; }
__host__ __device__ inline int st_z(int batch, int b) { return (batch + b) * 32; }
__host__ __device__ inline int st_mu(int batch) { return 2 * batch * 32; }
__host__ __device__ inline int st_rstd(int batch) { return 2 * batch * 32 + 32; }

// ------------------------------------------------------------------------------------------------ forward: attention + fold
// grid (ceil(co*ci/256), nconvs); every block recomputes the (tiny) attention of ALL samples, block x = 0 saves it.
__global__ void __launch_bounds__(256) osa_assemble_train_kernel(const __grid_constant__ OsaTrainLaunch L) {
  pdl_wait();
  pdl_trigger();
  const savsr_osa_params& c = L.c[blockIdx.y];
  const savsr_osa_train& tr = L.t[blockIdx.y];
  extern __shared__ float sm[];                       // zpre [B][32] | z [B][32] | att [B][nout]
  if (blockIdx.x * blockDim.x >= c.co * c.ci) return;
  const int B = L.batch;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int stride = osat_scratch_stride(c.ci);
  const int nout = c.ci + c.co + 9 + 8;
  float* zpre_s = sm;
  float* z_s = sm + B * 32;
  float* att_s = sm + 2 * B * 32;
  const bool saver = blockIdx.x == 0;
  for (int a = warp; a < c.att; a += 8) {
    float wr[10];
#pragma unroll
    for (int j = 0; j < 10; ++j) wr[j] = lane + 32 * j < c.ci ? __ldg(c.fc_w + a * c.ci + lane + 32 * j) : 0.f;
    float s1 = 0.f, s2 = 0.f;
    for (int n = 0; n < B; ++n) {
      const float* v2 = c.scratch + static_cast<long>(n) * stride + osat_off_v2(c.ci);
      float acc = 0.f;
#pragma unroll
      for (int j = 0; j < 10; ++j) if (lane + 32 * j < c.ci) acc += wr[j] * v2[lane + 32 * j];
#pragma unroll
      for (int off = 16; off >= 1; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
      if (lane == 0) zpre_s[n * 32 + a] = acc;
      s1 += acc;
    }
    const float mu = s1 / B;
    __syncwarp();
    for (int n = 0; n < B; ++n) { const float d = zpre_s[n * 32 + a] - mu; s2 += d * d; }
    const float var = s2 / B;                                  // biased variance normalises (F.batch_norm, training = True)
    const float rstd = rsqrtf(var + tr.eps);
    if (lane == 0) {
      const float gm = tr.bn_weight[a], bt = tr.bn_bias[a];
      for (int n = 0; n < B; ++n) z_s[n * 32 + a] = fmaxf((zpre_s[n * 32 + a] - mu) * rstd * gm + bt, 0.f);
      if (saver) {
        for (int n = 0; n < B; ++n) { tr.state[st_zpre(n) + a] = zpre_s[n * 32 + a]; tr.state[st_z(B, n) + a] = z_s[n * 32 + a]; }
        tr.state[st_mu(B) + a] = mu;
        tr.state[st_rstd(B) + a] = rstd;
        if (tr.running_mean) {                                  // running statistics: momentum update with the UNBIASED variance
          const float unb = B > 1 ? var * B / (B - 1) : var;
          tr.running_mean[a] = (1.f - tr.momentum) * tr.running_mean[a] + tr.momentum * mu;
          tr.running_var[a] = (1.f - tr.momentum) * tr.running_var[a] + tr.momentum * unb;
        }
      }
    }
  }
  __syncthreads();
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
    for (int n = 0; n < B; ++n) {
      float acc = b;
#pragma unroll
      for (int a = 0; a < 32; ++a) if (a < c.att) acc += wv[a] * z_s[n * 32 + a];
      att_s[n * nout + j] = sig ? sigmoid_t(acc) : acc;
    }
  }
  __syncthreads();
  if (threadIdx.x < B) {
    float* ka = att_s + threadIdx.x * nout + c.ci + c.co + 9;
    float mx = ka[0];
    for (int k = 1; k < 8; ++k) mx = fmaxf(mx, ka[k]);
    float e[8], sum = 0.f;
    for (int k = 0; k < 8; ++k) { e[k] = expf(ka[k] - mx); sum += e[k]; }
    for (int k = 0; k < 8; ++k) ka[k] = e[k] / sum;
  }
  __syncthreads();
  if (saver) {
    for (int r = threadIdx.x; r < B * nout; r += blockDim.x) {
      const int n = r / nout, j = r - n * nout;
      c.scratch[static_cast<long>(n) * stride + osat_off_att(c.ci) + j] = att_s[r];
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
  const int row = quad_row(o);
  const int inner = row * 64 + ((((kk >> 3) ^ (row & 7)) << 3) | (kk & 7));
  const int row_t = quad_row(kk);                              // transposed operand: rows = input channels, K = output channels
  const int inner_t = row_t * 64 + ((((o >> 3) ^ (row_t & 7)) << 3) | (o & 7));
  for (int n = 0; n < B; ++n) {
    const float* att = att_s + n * nout;
    const float ca = att[i], fa = att[c.ci + o];
    const float* sa = att + c.ci + c.co;
    const float* ka = sa + 9;
    uint16_t* dst = static_cast<uint16_t*>(c.packed) + n * sample_elems;                                   // [n][s][9][64][64]
    uint16_t* dst_t = static_cast<uint16_t*>(tr.packed_t) + (static_cast<long>(s) * B + n) * 9 * 4096;     // [s][n][9][64][64]
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      float acc = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) acc += ka[k] * bk[k][t];
      const uint16_t h = float_to_h(acc * sa[t] * ca * fa, L.fmt);
      dst[static_cast<long>(s * 9 + t) * 4096 + inner] = h;
      dst_t[(8 - t) * 4096 + inner_t] = h;
    }
  }
}

// ------------------------------------------------------------------------------------------------ backward 1: through the fold
// W'[b,o,i,t] = fa[b,o] ca[b,i] sa[b,t] M[b,o,i,t],  M = sum_k ka[b,k] bank[k,o,i,t].   grid (ci / 2, nconvs), 128 threads.
// Samples are processed four at a time (registers); dwfold is zeroed after it has been read (the next step's atomics start from 0).
__global__ void __launch_bounds__(128) osa_unfold_bwd_kernel(const __grid_constant__ OsaTrainLaunch L) {
  pdl_wait();
  pdl_trigger();
  const savsr_osa_params& c = L.c[blockIdx.y];
  const savsr_osa_grads& g = L.g[blockIdx.y];
  extern __shared__ float sm[];                       // att [B][nout] | part [4 warps][B][18]
  if (static_cast<int>(blockIdx.x) >= c.ci / 2) return;   // (ci / 16) x (64 / 8) blocks
  const int B = L.batch;
  const int nout = c.ci + c.co + 9 + 8;
  const int stride = osat_scratch_stride(c.ci);
  float* att_s = sm;
  float* part = sm + B * nout;
  for (int r = threadIdx.x; r < B * nout; r += blockDim.x) {
    const int n = r / nout, j = r - n * nout;
    att_s[r] = c.scratch[static_cast<long>(n) * stride + osat_off_att(c.ci) + j];
  }
  __syncthreads();
  // block = 16 input channels x 8 output channels, thread t = (o = t & 7, i = t >> 3): the bank (OIHW) is read as 144-byte runs and
  // dwfold ([tap][i][o]) as whole 32-byte sectors.  d ca reduces over the 8 lanes sharing i, d fa over the 4 lanes sharing o, d ka / d sa
  // over the block.  No shared-memory float atomics (they compile to CAS loops).
  const int ib = blockIdx.x % (c.ci / 16), ob = blockIdx.x / (c.ci / 16);
  const int i = ib * 16 + (threadIdx.x >> 3), o = ob * 8 + (threadIdx.x & 7);
  const long per_k = static_cast<long>(c.co) * c.ci * 9;
  const long pos = (static_cast<long>(o) * c.ci + i) * 9;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float bk[8][9];                                      // the 72 bank values of this filter position: all loads in flight at once
#pragma unroll
  for (int k = 0; k < 8; ++k) {
#pragma unroll
    for (int u = 0; u < 9; ++u) bk[k][u] = __ldg(c.bank + k * per_k + pos + u);
  }
  for (int b0 = 0; b0 < B; b0 += 4) {
    float t[4][9], fc[4];
#pragma unroll
    for (int bb = 0; bb < 4; ++bb) {
      const int b = b0 + bb;
      const bool ok = b < B;
      float* src = g.dwfold + b * per_k + static_cast<long>(i) * 64 + o;          // SAVSR_WGRAD_TIO: [b][tap][i][o]
      const long tap_stride = static_cast<long>(c.ci) * 64;
#pragma unroll
      for (int u = 0; u < 9; ++u) { t[bb][u] = ok ? src[u * tap_stride] : 0.f; if (ok) src[u * tap_stride] = 0.f; }
      fc[bb] = ok ? att_s[b * nout + i] * att_s[b * nout + c.ci + o] : 0.f;
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float db[9];
#pragma unroll
      for (int u = 0; u < 9; ++u) db[u] = 0.f;
#pragma unroll
      for (int bb = 0; bb < 4; ++bb) {
        const int b = b0 + bb;
        if (b >= B) continue;
        const float* sa = att_s + b * nout + c.ci + c.co;
        const float ka = sa[9 + k];
        float dka = 0.f;
#pragma unroll
        for (int u = 0; u < 9; ++u) {
          const float q = fc[bb] * sa[u] * t[bb][u];
          db[u] += ka * q;
          dka += q * bk[k][u];
        }
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) dka += __shfl_xor_sync(0xffffffffu, dka, off);
        if (lane == 0) part[(warp * B + b) * 18 + 9 + k] = dka;
      }
      float* dst = g.d_bank + k * per_k + pos;
#pragma unroll
      for (int u = 0; u < 9; ++u) dst[u] += db[u];
    }
#pragma unroll
    for (int bb = 0; bb < 4; ++bb) {
      const int b = b0 + bb;
      if (b >= B) continue;
      const float* sa = att_s + b * nout + c.ci + c.co;
      const float ca = att_s[b * nout + i], fa = att_s[b * nout + c.ci + o];
      float sp = 0.f;
#pragma unroll
      for (int u = 0; u < 9; ++u) {
        float Mu = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) Mu += sa[9 + k] * bk[k][u];
        const float P = t[bb][u] * Mu;
        sp += sa[u] * P;
        float ds = fa * ca * P;
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) ds += __shfl_xor_sync(0xffffffffu, ds, off);
        if (lane == 0) part[(warp * B + b) * 18 + u] = ds;
      }
      float dca = fa * sp;                                      // d ca[i]: the 8 lanes with the same i
#pragma unroll
      for (int off = 4; off >= 1; off >>= 1) dca += __shfl_xor_sync(0xffffffffu, dca, off);
      if ((lane & 7) == 0) atomicAdd(g.datt + b * nout + i, dca);
      float dfa = ca * sp;                                      // d fa[o]: the 4 lanes with the same o
      dfa += __shfl_xor_sync(0xffffffffu, dfa, 8);
      dfa += __shfl_xor_sync(0xffffffffu, dfa, 16);
      if (lane < 8) atomicAdd(g.datt + b * nout + c.ci + o, dfa);
    }
  }
  __syncthreads();
  for (int r = threadIdx.x; r < B * 17; r += blockDim.x) {      // d sa (9) and d ka (8) of the block
    const int b = r / 17, q = r - b * 17;
    float v = 0.f;
    for (int w = 0; w < 4; ++w) v += part[(w * B + b) * 18 + q];
    atomicAdd(g.datt + b * nout + c.ci + c.co + q, v);
  }
}

// ------------------------------------------------------------------------------------------------ backward 2: vectors
// One CTA (1024 threads) per convolution: heads -> ReLU -> BatchNorm (batch statistics) -> fc -> ReLU (the small layers); the two
// large scale_routing layers follow in osa_attn_matvec_kernel.
// Writes the vectors the weight-gradient kernel needs to g.dvec: dpre [B][nout] | dzpre [B][32] | dv2 [B][ci] | dh1 [B][2ci], the
// BatchNorm weight / bias gradients, and dpool [B][ci] (the gradient of the pooled means, already through routing.0).
__host__ __device__ inline int dv_dpre(int) { return 0; }
__host__ __device__ inline int dv_dzpre(int batch, int nout) { return batch * nout; }
__host__ __device__ inline int dv_dv2(int batch, int nout) { return batch * nout + batch * 32; }
__host__ __device__ inline int dv_dh1(int batch, int nout, int ci) { return batch * nout + batch * 32 + batch * ci; }
__host__ __device__ inline int dv_total(int batch, int nout, int ci) { return batch * nout + batch * 32 + 3 * batch * ci; }

__global__ void __launch_bounds__(1024) osa_attn_chain_kernel(const __grid_constant__ OsaTrainLaunch L) {
  pdl_wait();
  pdl_trigger();
  const savsr_osa_params& c = L.c[blockIdx.x];
  const savsr_osa_train& tr = L.t[blockIdx.x];
  const savsr_osa_grads& g = L.g[blockIdx.x];
  extern __shared__ float sm[];
  const int B = L.batch, ci = c.ci, att = c.att;
  const int nout = ci + c.co + 9 + 8;
  const int stride = osat_scratch_stride(ci);
  float* dpre = sm;                      // [B][nout]
  float* dzn = dpre + B * nout;          // [B][32]   (becomes dzpre)
  float* dv2 = dzn + B * 32;             // [B][ci]
  float* dh1 = dv2 + B * ci;             // [B][2ci]
  float* dot = dh1 + 2 * B * ci;         // [B]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // softmax: dot[b] = sum_k ka dka
  if (tid < B) {
    const float* a = c.scratch + static_cast<long>(tid) * stride + osat_off_att(ci) + ci + c.co + 9;
    const float* d = g.datt + tid * nout + ci + c.co + 9;
    float s = 0.f;
    for (int k = 0; k < 8; ++k) s += a[k] * d[k];
    dot[tid] = s;
  }
  __syncthreads();
  for (int r = tid; r < B * nout; r += blockDim.x) {
    const int b = r / nout, j = r - b * nout;
    const float a = c.scratch[static_cast<long>(b) * stride + osat_off_att(ci) + j];
    const float d = g.datt[r];
    g.datt[r] = 0.f;                                            // ready for the next step's atomics
    const float v = j < ci + c.co + 9 ? d * a * (1.f - a) : a * (d - dot[b]);
    dpre[r] = v;
    g.dvec[dv_dpre(0) + r] = v;
  }
  __syncthreads();
  // dz[b][a] = sum_j dpre[b][j] HW[j][a]; one warp per (b, a)
  for (int pr = warp; pr < B * att; pr += 32) {
    const int b = pr / att, a = pr - b * att;
    float acc = 0.f;
    for (int j = lane; j < nout; j += 32) {
      const float* w;
      if (j < ci) w = c.ch_w + j * att;
      else if (j < ci + c.co) w = c.fl_w + (j - ci) * att;
      else if (j < ci + c.co + 9) w = c.sp_w + (j - ci - c.co) * att;
      else w = c.kn_w + (j - ci - c.co - 9) * att;
      acc += dpre[b * nout + j] * __ldg(w + a);
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (lane == 0) dzn[b * 32 + a] = tr.state[st_z(B, b) + a] > 0.f ? acc : 0.f;
  }
  __syncthreads();
  if (tid < att) {                                             // BatchNorm backward over the batch, channel tid
    const int a = tid;
    const float mu = tr.state[st_mu(B) + a], rstd = tr.state[st_rstd(B) + a], gm = tr.bn_weight[a];
    float s1 = 0.f, s2 = 0.f;
    for (int b = 0; b < B; ++b) {
      const float xh = (tr.state[st_zpre(b) + a] - mu) * rstd;
      s1 += dzn[b * 32 + a];
      s2 += dzn[b * 32 + a] * xh;
    }
    g.d_bn_w[a] += s2;
    g.d_bn_b[a] += s1;
    for (int b = 0; b < B; ++b) {
      const float xh = (tr.state[st_zpre(b) + a] - mu) * rstd;
      const float v = gm * rstd * (dzn[b * 32 + a] - s1 / B - xh * s2 / B);
      dzn[b * 32 + a] = v;
      g.dvec[dv_dzpre(B, nout) + b * 32 + a] = v;
    }
  }
  __syncthreads();
  for (int r = tid; r < B * ci; r += blockDim.x) {             // dv2 = dzpre FC, through the ReLU of routing.2
    const int b = r / ci, i = r - b * ci;
    float acc = 0.f;
    for (int a = 0; a < att; ++a) acc += dzn[b * 32 + a] * __ldg(c.fc_w + a * ci + i);
    const float v = c.scratch[static_cast<long>(b) * stride + osat_off_v2(ci) + i] > 0.f ? acc : 0.f;
    dv2[r] = v;
    g.dvec[dv_dv2(B, nout) + r] = v;
  }
}

// out[b][col] = sum_row in[b][row] W[row][col] for the two large layers of scale_routing, many blocks per convolution:
//   layer 1: dh1 = dv2 R2 ([ci][2ci]), through the ReLU of routing.0 (mask h1 > 0), written to dvec;
//   layer 0: dvin = dh1 R0 ([2ci][ci+2]); columns 2.. are the pooled means -> dpool.
// grid (ceil(cols/32), nconvs), 512 threads: warp w sums the rows w, w+16, ... for 32 columns (coalesced), shared-memory reduce.
// NB: batch bucket (8, 16 or 32) >= B, the number of per-sample accumulators each thread keeps in registers.
template <int NB>
__global__ void __launch_bounds__(512) osa_attn_matvec_kernel(const __grid_constant__ OsaTrainLaunch L, int layer) {
  pdl_wait();
  pdl_trigger();
  const savsr_osa_params& c = L.c[blockIdx.y];
  const savsr_osa_grads& g = L.g[blockIdx.y];
  extern __shared__ float sm[];                       // red [16 warps][B][32] | in_s [B][rows], rows <= 640
  const int B = L.batch, ci = c.ci;
  const int nout = ci + c.co + 9 + 8;
  const int rows = layer == 1 ? ci : 2 * ci, cols = layer == 1 ? 2 * ci : ci + 2;
  if (blockIdx.x * 32 >= cols) return;
  float* red = sm;
  float* in_s = sm + 16 * B * 32;
  const float* W = layer == 1 ? c.r2_w : c.r0_w;
  const float* in = g.dvec + (layer == 1 ? dv_dv2(B, nout) : dv_dh1(B, nout, ci));
  for (int r = threadIdx.x; r < B * rows; r += blockDim.x) in_s[r] = in[r];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int col = blockIdx.x * 32 + lane;
  float acc[NB];
#pragma unroll
  for (int b = 0; b < NB; ++b) acc[b] = 0.f;
  if (col < cols) {
    int r = warp;
    for (; r + 48 < rows; r += 64) {                          // four independent weight loads in flight per warp
      float w[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) w[q] = __ldg(W + static_cast<long>(r + 16 * q) * cols + col);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
#pragma unroll
        for (int b = 0; b < NB; ++b) if (b < B) acc[b] += in_s[b * rows + r + 16 * q] * w[q];
      }
    }
    for (; r < rows; r += 16) {
      const float w = __ldg(W + static_cast<long>(r) * cols + col);
#pragma unroll
      for (int b = 0; b < NB; ++b) if (b < B) acc[b] += in_s[b * rows + r] * w;
    }
  }
#pragma unroll
  for (int b = 0; b < NB; ++b) if (b < B) red[(warp * B + b) * 32 + lane] = acc[b];
  __syncthreads();
  for (int b = threadIdx.x >> 5; b < B && col < cols; b += 16) {   // the warps finish one sample each (two at B > 16)
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < 16; ++w) v += red[(w * B + b) * 32 + lane];
    const int stride = osat_scratch_stride(ci);
    if (layer == 1) {
      g.dvec[dv_dh1(B, nout, ci) + b * 2 * ci + col] = c.scratch[static_cast<long>(b) * stride + osat_off_h1(ci) + col] > 0.f ? v : 0.f;
    } else if (col >= 2) {
      g.dpool[b * ci + (col - 2)] = v;
    }
  }
}

// ------------------------------------------------------------------------------------------------ backward 3: weight gradients
// dW[r][q] += sum_b dout[b][r] in[b][q] for the seven matrices of the prologue, biases likewise; grid (blocks, nconvs).
__global__ void __launch_bounds__(256) osa_attn_wgrad_kernel(const __grid_constant__ OsaTrainLaunch L) {
  pdl_wait();
  pdl_trigger();
  const savsr_osa_params& c = L.c[blockIdx.y];
  const savsr_osa_train& tr = L.t[blockIdx.y];
  const savsr_osa_grads& g = L.g[blockIdx.y];
  const int B = L.batch, ci = c.ci, att = c.att, co = c.co;
  const int nout = ci + co + 9 + 8;
  const int stride = osat_scratch_stride(ci);
  const float* dpre = g.dvec + dv_dpre(0);
  const float* dzpre = g.dvec + dv_dzpre(B, nout);
  const float* dv2 = g.dvec + dv_dv2(B, nout);
  const float* dh1 = g.dvec + dv_dh1(B, nout, ci);
  const long n_heads = static_cast<long>(nout) * att, n_fc = static_cast<long>(att) * ci, n_r2 = static_cast<long>(ci) * 2 * ci,
             n_r0 = 2L * ci * (ci + 2);
  const long total = n_heads + nout + n_fc + n_r2 + ci + n_r0 + 2 * ci;
  for (long e = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; e < total; e += static_cast<long>(gridDim.x) * blockDim.x) {
    long r = e;
    float acc = 0.f;
    float* dst;
    if (r < n_heads) {                                          // head weights [j][a] <- dpre[b][j] z[b][a]
      const int j = static_cast<int>(r / att), a = static_cast<int>(r - static_cast<long>(j) * att);
      for (int b = 0; b < B; ++b) acc += dpre[b * nout + j] * tr.state[st_z(B, b) + a];
      if (j < ci) dst = g.d_ch_w + j * att + a;
      else if (j < ci + co) dst = g.d_fl_w + (j - ci) * att + a;
      else if (j < ci + co + 9) dst = g.d_sp_w + (j - ci - co) * att + a;
      else dst = g.d_kn_w + (j - ci - co - 9) * att + a;
    } else if ((r -= n_heads) < nout) {                         // head biases
      const int j = static_cast<int>(r);
      for (int b = 0; b < B; ++b) acc += dpre[b * nout + j];
      if (j < ci) dst = g.d_ch_b + j;
      else if (j < ci + co) dst = g.d_fl_b + (j - ci);
      else if (j < ci + co + 9) dst = g.d_sp_b + (j - ci - co);
      else dst = g.d_kn_b + (j - ci - co - 9);
    } else if ((r -= nout) < n_fc) {                            // fc [a][i] <- dzpre[b][a] v2[b][i]
      const int a = static_cast<int>(r / ci), i = static_cast<int>(r - static_cast<long>(a) * ci);
      for (int b = 0; b < B; ++b) acc += dzpre[b * 32 + a] * c.scratch[static_cast<long>(b) * stride + osat_off_v2(ci) + i];
      dst = g.d_fc_w + r;
    } else if ((r -= n_fc) < n_r2) {                            // routing.2 [i][j] <- dv2[b][i] h1[b][j]
      const int i = static_cast<int>(r / (2 * ci)), j = static_cast<int>(r - static_cast<long>(i) * 2 * ci);
      for (int b = 0; b < B; ++b) acc += dv2[b * ci + i] * c.scratch[static_cast<long>(b) * stride + osat_off_h1(ci) + j];
      dst = g.d_r2_w + r;
    } else if ((r -= n_r2) < ci) {
      for (int b = 0; b < B; ++b) acc += dv2[b * ci + r];
      dst = g.d_r2_b + r;
    } else if ((r -= ci) < n_r0) {                              // routing.0 [j][m] <- dh1[b][j] vin[b][m]
      const int j = static_cast<int>(r / (ci + 2)), m = static_cast<int>(r - static_cast<long>(j) * (ci + 2));
      for (int b = 0; b < B; ++b) acc += dh1[b * 2 * ci + j] * c.scratch[static_cast<long>(b) * stride + m];
      dst = g.d_r0_w + r;
    } else {
      r -= n_r0;
      for (int b = 0; b < B; ++b) acc += dh1[b * 2 * ci + r];
      dst = g.d_r0_b + r;
    }
    *dst += acc;
  }
}

// ------------------------------------------------------------------------------------------------ RCAB channel attention backward
// dy[n][c] = sum_p dout[n,p,c] t[n,p,c] on two arena slots.  grid (blocks, batch), 256 threads; out must be zero on entry.
__global__ void __launch_bounds__(256) slot_channel_dot_kernel(const uint16_t* __restrict__ a, const uint16_t* __restrict__ b, float* __restrict__ out,
                                                               long npix, int fmt) {
  pdl_wait();
  pdl_trigger();
  __shared__ float red[64];
  const int n = blockIdx.y;
  if (threadIdx.x < 64) red[threadIdx.x] = 0.f;
  __syncthreads();
  const uint4* aa = reinterpret_cast<const uint4*>(a + static_cast<long>(n) * npix * kC);
  const uint4* bb = reinterpret_cast<const uint4*>(b + static_cast<long>(n) * npix * kC);
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  const long chunks = npix * 8;
  // the stride (gridDim.x * 256) is a multiple of 8, so a thread always sees the same 8-channel group
  for (long id = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; id < chunks; id += static_cast<long>(gridDim.x) * blockDim.x) {
    const uint4 x = aa[id], y = bb[id];
    acc[0] += h_lo(x.x, fmt) * h_lo(y.x, fmt); acc[1] += h_hi(x.x, fmt) * h_hi(y.x, fmt);
    acc[2] += h_lo(x.y, fmt) * h_lo(y.y, fmt); acc[3] += h_hi(x.y, fmt) * h_hi(y.y, fmt);
    acc[4] += h_lo(x.z, fmt) * h_lo(y.z, fmt); acc[5] += h_hi(x.z, fmt) * h_hi(y.z, fmt);
    acc[6] += h_lo(x.w, fmt) * h_lo(y.w, fmt); acc[7] += h_hi(x.w, fmt) * h_hi(y.w, fmt);
  }
  const int c0 = (threadIdx.x & 7) * 8;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float v = acc[j];
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 16);
    if ((threadIdx.x & 31) < 8) atomicAdd(&red[c0 + j], v);
  }
  __syncthreads();
  if (threadIdx.x < 64) atomicAdd(out + n * 64 + threadIdx.x, red[threadIdx.x]);
}

struct CaBwdParams {
  const float* pool; int npart; float inv_npix;
  const float *w1, *b1, *w2, *b2;
  float* dy;            // [B][64] in, zeroed on exit
  const float* y;       // [B][64] saved sigmoid output
  float *dw1, *db1, *dw2, *db2;
  float* dmean;         // [B][64] out
  int batch;
};
// one CTA, 1024 threads: the pooled partial sums are reduced by 16 ranges x 64 channels with all loads in flight, the rest is tiny
__global__ void __launch_bounds__(1024) ca_backward_kernel(const CaBwdParams p) {
  pdl_wait();
  pdl_trigger();
  const int tid = threadIdx.x;
  const int B = p.batch;
  extern __shared__ float sm[];                       // part [16][B][64] | mean [B][64] | ds [B][64] | hid [B][4] | dhid [B][4]
  float* part = sm;
  float* mean = part + 16 * B * 64;
  float* ds = mean + B * 64;
  float* hid = ds + B * 64;
  float* dhid = hid + B * 4;
  {
    const int c = tid & 63, q16 = tid >> 6;
    for (int n = 0; n < B; ++n) {
      const float* src = p.pool + static_cast<long>(n) * p.npart * kC;
      float a[4] = {0.f, 0.f, 0.f, 0.f};
      int q = q16;
      for (; q + 48 < p.npart; q += 64) {
#pragma unroll
        for (int j = 0; j < 4; ++j) a[j] += src[(q + 16 * j) * kC + c];
      }
      for (; q < p.npart; q += 16) a[0] += src[q * kC + c];
      part[(q16 * B + n) * 64 + c] = (a[0] + a[1]) + (a[2] + a[3]);
    }
  }
  __syncthreads();
  for (int r = tid; r < B * 64; r += blockDim.x) {
    const int n = r >> 6, c = r & 63;
    float m = 0.f;
#pragma unroll
    for (int q = 0; q < 16; ++q) m += part[(q * B + n) * 64 + c];
    mean[r] = m * p.inv_npix;
    const float yy = p.y[r];
    ds[r] = p.dy[r] * yy * (1.f - yy);
    p.dy[r] = 0.f;
  }
  __syncthreads();
  if (tid < B * 4) {
    const int n = tid >> 2, k = tid & 3;
    float a = p.b1[k], d = 0.f;
    for (int c = 0; c < 64; ++c) { a += p.w1[k * 64 + c] * mean[n * 64 + c]; d += p.w2[c * 4 + k] * ds[n * 64 + c]; }
    hid[tid] = fmaxf(a, 0.f);
    dhid[tid] = a > 0.f ? d : 0.f;
  }
  __syncthreads();
  if (tid < 256) {                                             // weight gradients: 256 threads = w2 [64][4] and w1 [4][64]
    const int c = tid >> 2, k = tid & 3;
    float a2 = 0.f, a1 = 0.f;
    for (int n = 0; n < B; ++n) { a2 += ds[n * 64 + c] * hid[n * 4 + k]; a1 += dhid[n * 4 + k] * mean[n * 64 + c]; }
    p.dw2[c * 4 + k] += a2;
    p.dw1[k * 64 + c] += a1;
    if (tid < 64) { float s = 0.f; for (int n = 0; n < B; ++n) s += ds[n * 64 + tid]; p.db2[tid] += s; }
    if (tid < 4) { float s = 0.f; for (int n = 0; n < B; ++n) s += dhid[n * 4 + tid]; p.db1[tid] += s; }
  }
  for (int r = tid; r < B * 64; r += blockDim.x) {
    const int n = r >> 6, c = r & 63;
    float a = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) a += p.w1[k * 64 + c] * dhid[n * 4 + k];
    p.dmean[r] = a;
  }
}

}  // namespace savsr

using namespace savsr;

// defined in small_ops.cu: the pooling + scale_routing launches shared with the inference prologue
namespace savsr { int osa_prologue_front(savsr_ctx* ctx, const savsr_osa_params* convs, int nconvs, int batch, int npart, int npix, float inv_scale_h,
                                         float inv_scale_w, cudaStream_t st); }

// Dynamic shared memory of each kernel (bytes) for `batch` samples and a largest input width of `ci` channels (nout = ci + 64 + 17);
// the attribute of each kernel is raised once per context to its size at kMaxBatchT samples and ci = 64 * SAVSR_MAX_SRC.
constexpr size_t smem_assemble(int batch, int ci) { return (2 * 32 + static_cast<size_t>(ci + 81)) * batch * sizeof(float); }
constexpr size_t smem_unfold(int batch, int ci) { return (static_cast<size_t>(ci + 81) + 4 * 18) * batch * sizeof(float); }
constexpr size_t smem_chain(int batch, int ci) { return (static_cast<size_t>(ci + 81) + 32 + 3 * static_cast<size_t>(ci) + 1) * batch * sizeof(float); }
constexpr size_t smem_matvec(int batch, int ci) { return (16 * 32 + 2 * static_cast<size_t>(ci)) * batch * sizeof(float); }
constexpr size_t smem_ca_backward(int batch) { return (16 * 64 + 2 * 64 + 2 * 4) * static_cast<size_t>(batch) * sizeof(float); }
constexpr int kCiMaxT = 64 * SAVSR_MAX_SRC;
static_assert(smem_assemble(kMaxBatchT, kCiMaxT) <= 227 * 1024 && smem_unfold(kMaxBatchT, kCiMaxT) <= 227 * 1024 &&
              smem_chain(kMaxBatchT, kCiMaxT) <= 227 * 1024 && smem_matvec(kMaxBatchT, kCiMaxT) <= 227 * 1024 &&
              smem_ca_backward(kMaxBatchT) <= 227 * 1024, "kMaxBatchT samples exceed the 227 KB of shared memory a block may use");

static int fill_launch(const char* who, OsaTrainLaunch& L, savsr_ctx* ctx, const savsr_osa_params* convs, const savsr_osa_train* extra,
                       const savsr_osa_grads* grads, int nconvs, int batch) {
  SAVSR_REQUIRE(ctx && convs && extra, "%s: null pointer", who);
  SAVSR_REQUIRE(nconvs >= 1 && nconvs <= kMaxOsaT, "%s: nconvs %d out of range [1,%d]", who, nconvs, kMaxOsaT);
  SAVSR_REQUIRE(batch >= 1 && batch <= kMaxBatchT, "%s: batch %d out of range [1,%d]", who, batch, kMaxBatchT);
  memset(&L, 0, sizeof(L));
  for (int i = 0; i < nconvs; ++i) {
    const savsr_osa_params& c = convs[i];
    SAVSR_REQUIRE(c.ci > 0 && c.ci % 64 == 0 && c.ci <= 64 * SAVSR_MAX_SRC && c.co == 64 && c.att > 0 && c.att <= 32, "%s: conv %d shape unsupported", who, i);
    SAVSR_REQUIRE(c.bank && c.r0_w && c.r0_b && c.r2_w && c.r2_b && c.fc_w && c.ch_w && c.ch_b && c.fl_w && c.fl_b && c.sp_w && c.sp_b && c.kn_w &&
                  c.kn_b && c.scratch && c.packed, "%s: conv %d has a null parameter pointer", who, i);
    SAVSR_REQUIRE(extra[i].bn_weight && extra[i].bn_bias && extra[i].state && extra[i].packed_t, "%s: conv %d has a null train-mode pointer", who, i);
    L.c[i] = c;
    L.t[i] = extra[i];
    if (grads) {
      const savsr_osa_grads& g = grads[i];
      SAVSR_REQUIRE(g.dwfold && g.d_bank && g.d_r0_w && g.d_r0_b && g.d_r2_w && g.d_r2_b && g.d_fc_w && g.d_bn_w && g.d_bn_b && g.d_ch_w && g.d_ch_b &&
                    g.d_fl_w && g.d_fl_b && g.d_sp_w && g.d_sp_b && g.d_kn_w && g.d_kn_b && g.datt && g.dvec && g.dpool,
                    "%s: conv %d has a null gradient pointer", who, i);
      L.g[i] = g;
    }
  }
  L.nconvs = nconvs; L.batch = batch; L.fmt = ctx->fmt;
  return 0;
}

extern "C" int savsr_osa_prologue_train(savsr_ctx* ctx, const savsr_osa_params* convs, const savsr_osa_train* extra, int nconvs, int batch,
                                        int npart, int npix, float inv_scale_h, float inv_scale_w, savsr_stream st_) {
  OsaTrainLaunch L;
  if (int rc = fill_launch("savsr_osa_prologue_train", L, ctx, convs, extra, nullptr, nconvs, batch)) return rc;
  DeviceGuard guard(ctx->device);
  cudaStream_t st = static_cast<cudaStream_t>(st_);
  for (int i = 0; i < nconvs; ++i)
    for (int s = 0; s < convs[i].ci / 64; ++s) SAVSR_REQUIRE(convs[i].pool[s], "savsr_osa_prologue_train: conv %d source %d has no pool buffer", i, s);
  if (int rc = osa_prologue_front(ctx, convs, nconvs, batch, npart, npix, inv_scale_h, inv_scale_w, st)) return rc;
  int max_ci = 0;
  for (int i = 0; i < nconvs; ++i) max_ci = convs[i].ci > max_ci ? convs[i].ci : max_ci;
  const size_t smem = smem_assemble(batch, max_ci);
  if (smem > 48 * 1024) {
    if (int rc = ensure_smem_attr(ctx, kAttrOsaAssembleTrain, osa_assemble_train_kernel, smem_assemble(kMaxBatchT, kCiMaxT))) return rc;
  }
  (void)launch_k(ctx->opt[SAVSR_OPT_PDL] != 0, osa_assemble_train_kernel, dim3((64 * max_ci + 255) / 256, nconvs), dim3(256), smem, st, L);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

extern "C" size_t savsr_osa_train_state_floats(int batch) { return static_cast<size_t>(2 * batch + 2) * 32; }
extern "C" size_t savsr_osa_train_dvec_floats(int batch, int ci) { return static_cast<size_t>(dv_total(batch, ci + 64 + 17, ci)); }

extern "C" int savsr_osa_fold_backward(savsr_ctx* ctx, const savsr_osa_params* convs, const savsr_osa_train* extra, const savsr_osa_grads* grads,
                                       int nconvs, int batch, savsr_stream st_) {
  OsaTrainLaunch L;
  SAVSR_REQUIRE(grads, "savsr_osa_fold_backward: null pointer");
  if (int rc = fill_launch("savsr_osa_fold_backward", L, ctx, convs, extra, grads, nconvs, batch)) return rc;
  DeviceGuard guard(ctx->device);
  cudaStream_t st = static_cast<cudaStream_t>(st_);
  int max_ci = 0;
  for (int i = 0; i < nconvs; ++i) max_ci = convs[i].ci > max_ci ? convs[i].ci : max_ci;
  const size_t smem1 = smem_unfold(batch, max_ci);
  if (smem1 > 48 * 1024) {
    if (int rc = ensure_smem_attr(ctx, kAttrOsaUnfoldBwd, osa_unfold_bwd_kernel, smem_unfold(kMaxBatchT, kCiMaxT))) return rc;
  }
  (void)launch_k(ctx->opt[SAVSR_OPT_PDL] != 0, osa_unfold_bwd_kernel, dim3(max_ci / 2, nconvs), dim3(128), smem1, st, L);
  const size_t smem2 = smem_chain(batch, max_ci);
  if (smem2 > 48 * 1024) {
    if (int rc = ensure_smem_attr(ctx, kAttrOsaChain, osa_attn_chain_kernel, smem_chain(kMaxBatchT, kCiMaxT))) return rc;
  }
  (void)launch_k(ctx->opt[SAVSR_OPT_PDL] != 0, osa_attn_chain_kernel, dim3(nconvs), dim3(1024), smem2, st, L);
  // the smallest batch bucket that holds the batch: b <= 8 keeps eight accumulators per thread
  void (*matvec)(const OsaTrainLaunch, int) = osa_attn_matvec_kernel<32>;
  int matvec_bit = kAttrOsaMatvec + 2;
  if (batch <= 8) { matvec = osa_attn_matvec_kernel<8>; matvec_bit = kAttrOsaMatvec; }
  else if (batch <= 16) { matvec = osa_attn_matvec_kernel<16>; matvec_bit = kAttrOsaMatvec + 1; }
  const size_t smem3 = smem_matvec(batch, max_ci);
  if (smem3 > 48 * 1024) {
    if (int rc = ensure_smem_attr(ctx, matvec_bit, matvec, smem_matvec(kMaxBatchT, kCiMaxT))) return rc;
  }
  (void)launch_k(ctx->opt[SAVSR_OPT_PDL] != 0, matvec, dim3((2 * max_ci + 31) / 32, nconvs), dim3(512), smem3, st, L, 1);
  (void)launch_k(ctx->opt[SAVSR_OPT_PDL] != 0, matvec, dim3((max_ci + 2 + 31) / 32, nconvs), dim3(512), smem3, st, L, 0);
  (void)launch_k(ctx->opt[SAVSR_OPT_PDL] != 0, osa_attn_wgrad_kernel, dim3(2 * ctx->sm_count / nconvs + 1, nconvs), dim3(256), 0, st, L);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int savsr_slot_channel_dot(savsr_ctx* ctx, savsr_arena* arena, int a_slot, int b_slot, float* out, savsr_stream st) {
  SAVSR_REQUIRE(ctx && arena && out, "savsr_slot_channel_dot: null pointer");
  SAVSR_REQUIRE(a_slot >= 0 && a_slot < arena->nslots && b_slot >= 0 && b_slot < arena->nslots, "savsr_slot_channel_dot: slot out of range");
  DeviceGuard guard(ctx->device);
  const long npix = static_cast<long>(arena->height) * arena->width;
  const long img = npix * kC * arena->batch;
  long blocks = (npix * 8 + 255) / 256;
  const long cap = 2L * ctx->sm_count / arena->batch + 1;
  if (blocks > cap) blocks = cap;
  (void)launch_k(ctx->opt[SAVSR_OPT_PDL] != 0, slot_channel_dot_kernel, dim3(static_cast<unsigned>(blocks), arena->batch), dim3(256), 0, static_cast<cudaStream_t>(st), 
      reinterpret_cast<const uint16_t*>(arena->base) + a_slot * img, reinterpret_cast<const uint16_t*>(arena->base) + b_slot * img, out, npix, ctx->fmt);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int savsr_ca_backward(savsr_ctx* ctx, const float* pool, int npart, int npix, int batch, const float* w1, const float* b1, const float* w2,
                                 const float* b2, const float* y, float* dy, float* dw1, float* db1, float* dw2, float* db2, float* dmean,
                                 savsr_stream st) {
  SAVSR_REQUIRE(ctx && pool && w1 && b1 && w2 && b2 && y && dy && dw1 && db1 && dw2 && db2 && dmean, "savsr_ca_backward: null pointer");
  SAVSR_REQUIRE(batch >= 1 && batch <= kMaxBatchT, "savsr_ca_backward: batch %d out of range [1,%d]", batch, kMaxBatchT);
  DeviceGuard guard(ctx->device);
  CaBwdParams p;
  p.pool = pool; p.npart = npart; p.inv_npix = 1.f / static_cast<float>(npix);
  p.w1 = w1; p.b1 = b1; p.w2 = w2; p.b2 = b2; p.dy = dy; p.y = y; p.dw1 = dw1; p.db1 = db1; p.dw2 = dw2; p.db2 = db2; p.dmean = dmean; p.batch = batch;
  const size_t smem = smem_ca_backward(batch);
  if (smem > 48 * 1024) {
    if (int rc = ensure_smem_attr(ctx, kAttrCaBackward, ca_backward_kernel, smem_ca_backward(kMaxBatchT))) return rc;
  }
  (void)launch_k(ctx->opt[SAVSR_OPT_PDL] != 0, ca_backward_kernel, dim3(1), dim3(1024), smem, static_cast<cudaStream_t>(st), p);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}
