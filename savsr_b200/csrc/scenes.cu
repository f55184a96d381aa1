// Scene cuts in a streamed video, resolved on the device.
//
// scene_score: the cut score of ring frame t against frame t - 1, in integers so that the device, a NumPy reference and the 8- and
// 16-bit rings agree exactly:
//   SAD_t = sum over all 3hw samples of |ring[t] - ring[t - 1]|  (uint64; SAD_0 = 0, frame 0 has no predecessor)
//   m_t   = min(SAD_t, |SAD_t - SAD_{t-1}|)                     (ffmpeg scdet's min(mafd, |mafd - prev_mafd|), scaled)
//   frame t >= 1 starts a shot when 100 m_t >= tau * 3hw * maxval, i.e. m_t >= bound = ceil(tau * 3hw * maxval / 100) (the host
//   computes it from the exact value of tau).
// One launch per frame: every block sums its share of |a - b| into a uint64 partial, and the last block to finish (a ticket counter in
// the caller's scratch) adds the partials and writes the cut flag and SAD_t into per-slot arrays.  Integer sums: the result does not
// depend on the order in which blocks finish.
//
// write_scene_frame_table: the frame table of a batch of windows, folded at the cuts the flags mark, without the host knowing them.
// The window of frame c reads frames c - 3 .. c + 3, so only the flags of frames c - 2 .. c + 3 can change it: the shot's start is the
// last flagged frame of c - 2 .. c (else max(c - 3, 0)), its end the first flagged frame of c + 1 .. c + 3 (else c + 4, or the number of
// frames once the end of the stream is known).  A shot of 4 or more frames folds as the single reflection at its ends, which only
// depends on the end that is within the window, so these bounds give the windows the true shot bounds give
// (savsr_b200/sharding.py: scene_window_indices).
#include "common.cuh"

namespace savsr {

constexpr int kSceneThreads = 256;
constexpr int kSceneMaxBlocks = SAVSR_SCENE_SCRATCH_WORDS - 1;

__device__ __forceinline__ unsigned sad16(uint4 a, uint4 b, uint8_t) {
  return __vsadu4(a.x, b.x) + __vsadu4(a.y, b.y) + __vsadu4(a.z, b.z) + __vsadu4(a.w, b.w);
}
__device__ __forceinline__ unsigned sad_u16x2(unsigned a, unsigned b) {
  const unsigned d = __vabsdiffu2(a, b);
  return (d & 0xffffu) + (d >> 16);
}
__device__ __forceinline__ unsigned sad16(uint4 a, uint4 b, uint16_t) {
  return sad_u16x2(a.x, b.x) + sad_u16x2(a.y, b.y) + sad_u16x2(a.z, b.z) + sad_u16x2(a.w, b.w);
}

__device__ __forceinline__ unsigned long long block_sum(unsigned long long v, unsigned long long* sh) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) sh[warp] = v;
  __syncthreads();
  unsigned long long s = 0;
  if (threadIdx.x == 0)
    for (int i = 0; i < kSceneThreads / 32; ++i) s += sh[i];
  __syncthreads();
  return s;   // valid in thread 0
}

// cur, prev: frames t and t - 1 (n samples each); vec: both 16-byte aligned, read as uint4 with a scalar tail.
template <typename T>
__global__ void __launch_bounds__(kSceneThreads) scene_score_kernel(const T* __restrict__ cur, const T* __restrict__ prev, long long n, int vec,
                                                                    long long t, int marked, unsigned long long bound, int slot, int prev_slot,
                                                                    uint8_t* __restrict__ cut, unsigned long long* __restrict__ sad,
                                                                    unsigned long long* __restrict__ scratch) {
  __shared__ unsigned long long sh[kSceneThreads / 32];
  __shared__ int last;
  unsigned long long acc = 0;
  if (t > 0) {
    const long long stride = static_cast<long long>(gridDim.x) * kSceneThreads;
    long long i0 = static_cast<long long>(blockIdx.x) * kSceneThreads + threadIdx.x;
    long long done = 0;
    if (vec) {
      constexpr int kPer = 16 / sizeof(T);
      const long long nv = n / kPer;
      const uint4* a = reinterpret_cast<const uint4*>(cur);
      const uint4* b = reinterpret_cast<const uint4*>(prev);
      for (long long i = i0; i < nv; i += stride) acc += sad16(__ldg(a + i), __ldg(b + i), T());
      done = nv * kPer;
    }
    for (long long i = done + i0; i < n; i += stride) {
      const int x = cur[i], y = prev[i];
      acc += static_cast<unsigned>(x > y ? x - y : y - x);
    }
  }
  const unsigned long long part = block_sum(acc, sh);
  if (threadIdx.x == 0) {
    scratch[1 + blockIdx.x] = part;
    __threadfence();
    last = atomicAdd(scratch, 1ull) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  unsigned long long s = 0;
  for (int i = threadIdx.x; i < static_cast<int>(gridDim.x); i += kSceneThreads) s += __ldcg(scratch + 1 + i);
  s = block_sum(s, sh);
  if (threadIdx.x == 0) {
    const unsigned long long before = t > 0 ? sad[prev_slot] : 0ull;
    const unsigned long long d = s > before ? s - before : before - s;
    const unsigned long long m = s < d ? s : d;
    cut[slot] = static_cast<uint8_t>((t > 0 && m >= bound) || marked);
    sad[slot] = s;
    scratch[0] = 0;   // the ticket counter is ready for the next frame's launch
  }
}

// One thread per table entry: window (entry / 7) of centre first + entry / 7, offset entry % 7 - 3.
__global__ void __launch_bounds__(256) write_scene_frame_table_kernel(const uint8_t** __restrict__ table, const uint8_t* ring, long long frame_bytes,
                                                                      int R, const uint8_t* __restrict__ cut, long long first, int count,
                                                                      long long received, int finished) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= count * 7) return;
  const long long c = first + e / 7, i = c + e % 7 - 3;
  long long start = c - 3 > 0 ? c - 3 : 0;
  for (long long f = c - 2; f <= c; ++f)
    if (f >= 1 && cut[f % R]) start = f;
  long long stop = c + 4;
  if (finished && received < stop) stop = received;
  for (long long f = c + 3; f > c; --f)
    if (f < received && cut[f % R]) stop = f;
  const long long L = stop - start;
  long long r = 0;
  if (L > 1) {
    const long long p = 2 * (L - 1);
    r = (i - start) % p;
    if (r < 0) r += p;
    if (r >= L) r = p - r;
  }
  table[e] = ring + ((start + r) % R) * frame_bytes;
}

template <typename T>
static int scene_score(const char* fn, savsr_ctx* ctx, const T* ring, int R, int h, int w, long long t, int marked, long long bound, uint8_t* cut,
                       unsigned long long* sad, unsigned long long* scratch, savsr_stream st) {
  SAVSR_REQUIRE(ctx && ring && cut && sad && scratch, "%s: null pointer (ctx, ring, cut, sad and scratch are all required)", fn);
  SAVSR_REQUIRE(R >= 7, "%s: ring of R = %d frames; a 7-frame window needs R >= 7", fn, R);
  SAVSR_REQUIRE(h > 0 && w > 0, "%s: bad frame size h=%d w=%d", fn, h, w);
  SAVSR_REQUIRE(t >= 0, "%s: frame index t = %lld is negative", fn, t);
  SAVSR_REQUIRE(bound > 0, "%s: threshold bound = %lld must be positive", fn, bound);
  DeviceGuard guard(ctx->device);
  const long long n = 3LL * h * w;
  const T* cur = ring + (t % R) * n;
  const T* prev = ring + ((t + R - 1) % R) * n;
  const int vec = ((reinterpret_cast<uintptr_t>(cur) | reinterpret_cast<uintptr_t>(prev)) & 15) == 0;
  const long long units = vec ? n / (16 / static_cast<long long>(sizeof(T))) : n;
  long long blocks = (units + kSceneThreads - 1) / kSceneThreads;
  const long long cap = 2LL * ctx->sm_count < kSceneMaxBlocks ? 2LL * ctx->sm_count : kSceneMaxBlocks;
  blocks = t == 0 ? 1 : (blocks < 1 ? 1 : (blocks > cap ? cap : blocks));
  scene_score_kernel<T><<<static_cast<unsigned>(blocks), kSceneThreads, 0, static_cast<cudaStream_t>(st)>>>(
      cur, prev, n, vec, t, marked != 0, static_cast<unsigned long long>(bound), static_cast<int>(t % R), static_cast<int>((t + R - 1) % R), cut,
      sad, scratch);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace savsr

using namespace savsr;

extern "C" int savsr_scene_score_u8(savsr_ctx* ctx, const uint8_t* ring, int R, int h, int w, long long t, int marked, long long bound, uint8_t* cut,
                                    unsigned long long* sad, unsigned long long* scratch, savsr_stream st) {
  return scene_score("savsr_scene_score_u8", ctx, ring, R, h, w, t, marked, bound, cut, sad, scratch, st);
}

extern "C" int savsr_scene_score_u16(savsr_ctx* ctx, const uint16_t* ring, int R, int h, int w, long long t, int marked, long long bound,
                                     uint8_t* cut, unsigned long long* sad, unsigned long long* scratch, savsr_stream st) {
  return scene_score("savsr_scene_score_u16", ctx, ring, R, h, w, t, marked, bound, cut, sad, scratch, st);
}

extern "C" int savsr_write_scene_frame_table(savsr_ctx* ctx, const uint8_t** table_dev, const void* ring, long long frame_bytes, int R,
                                             const uint8_t* cut, long long first, int count, long long received, int finished, savsr_stream st) {
  const char* fn = "savsr_write_scene_frame_table";
  SAVSR_REQUIRE(ctx && table_dev && ring && cut, "%s: null pointer (ctx, table_dev, ring and cut are all required)", fn);
  SAVSR_REQUIRE(R >= 7, "%s: ring of R = %d frames; a 7-frame window needs R >= 7", fn, R);
  SAVSR_REQUIRE(frame_bytes > 0, "%s: frame_bytes = %lld must be positive", fn, frame_bytes);
  SAVSR_REQUIRE(count >= 1 && first >= 0, "%s: bad batch: first = %lld, count = %d", fn, first, count);
  SAVSR_REQUIRE(finished == 0 || finished == 1, "%s: finished = %d must be 0 or 1", fn, finished);
  SAVSR_REQUIRE(first + count <= received, "%s: count = %d from first = %lld reaches past the %lld received frames", fn, count, first, received);
  SAVSR_REQUIRE(finished || first + count + 2 < received,
                "%s: count = %d from first = %lld: the last window reads frame %lld, but only %lld frames were received and the end of the "
                "stream is not known", fn, count, first, first + count + 2, received);
  const long long oldest = first - 3 > 0 ? first - 3 : 0;
  SAVSR_REQUIRE(received - oldest <= R, "%s: the windows read frames %lld .. %lld, more than the ring's R = %d slots hold", fn, oldest,
                received - 1, R);
  DeviceGuard guard(ctx->device);
  const int entries = count * 7;
  write_scene_frame_table_kernel<<<(entries + 255) / 256, 256, 0, static_cast<cudaStream_t>(st)>>>(
      table_dev, static_cast<const uint8_t*>(ring), frame_bytes, R, cut, first, count, received, finished);
  SAVSR_CUDA(cudaGetLastError());
  return 0;
}
