// savsr_plan: the forward as ONE C call (SURVEY.md section 8b: "savsr_forward(plan, x, scale, out, stream) once assembled").
// A plan is an ordered list of recorded launches -- the same entry points the host would call one by one, with their argument
// structures copied at record time -- replayed on a stream by savsr_plan_run.  It owns no device memory: arenas, weights, scratch and
// the I/O staging buffers stay the caller's (savsr_b200/engine.py builds them per (batch, h, w, scale) and records the list once).
// Replay is graph-capturable like every direct launch; a non-Python caller needs nothing but this header to run SAVSR.forward
// (lbasicsr/archs/savsr_arch.py:692-742) on prepared buffers.
#include <functional>
#include <vector>

#include "common.cuh"

struct savsr_plan {
  savsr_ctx* ctx;
  std::vector<std::function<int(savsr_stream)>> ops;
  void* x_in = nullptr;
  void* out = nullptr;
  size_t x_bytes = 0, out_bytes = 0;
  int format = SAVSR_FMT_BF16;
  bool u8 = false;                 // I/O mode: fp32 (savsr_forward) or uint8 BGR (savsr_forward_u8)
};

using namespace savsr;

extern "C" int savsr_plan_create(savsr_ctx* ctx, savsr_plan** out) {
  SAVSR_REQUIRE(ctx && out, "savsr_plan_create: null pointer");
  savsr_plan* p = new (std::nothrow) savsr_plan();
  SAVSR_REQUIRE(p, "savsr_plan_create: out of host memory");
  p->ctx = ctx;
  p->format = ctx->fmt;
  *out = p;
  return 0;
}
extern "C" void savsr_plan_destroy(savsr_plan* plan) { delete plan; }
extern "C" int savsr_plan_size(const savsr_plan* plan) { return plan ? static_cast<int>(plan->ops.size()) : 0; }

static int set_io(const char* name, savsr_plan* plan, void* x_in, size_t x_bytes, void* out, size_t out_bytes, int format, bool u8) {
  SAVSR_REQUIRE(plan && x_in && out && x_bytes && out_bytes, "%s: null pointer / empty buffer", name);
  SAVSR_REQUIRE(format == SAVSR_FMT_BF16 || format == SAVSR_FMT_FP16, "%s: unknown format %d", name, format);
  plan->x_in = x_in; plan->x_bytes = x_bytes; plan->out = out; plan->out_bytes = out_bytes; plan->format = format; plan->u8 = u8;
  return 0;
}

extern "C" int savsr_plan_set_io(savsr_plan* plan, float* x_in, size_t x_bytes, float* out, size_t out_bytes, int format) {
  return set_io("savsr_plan_set_io", plan, x_in, x_bytes, out, out_bytes, format, false);
}

extern "C" int savsr_plan_set_io_u8(savsr_plan* plan, uint8_t* x_in, size_t x_bytes, uint8_t* out, size_t out_bytes, int format) {
  return set_io("savsr_plan_set_io_u8", plan, x_in, x_bytes, out, out_bytes, format, true);
}

extern "C" int savsr_plan_add_pack_frames(savsr_plan* plan, savsr_arena* arena, const float* x, int t, int h, int w, int dst_slot) {
  SAVSR_REQUIRE(plan && arena && x, "savsr_plan_add_pack_frames: null pointer");
  savsr_ctx* ctx = plan->ctx;
  plan->ops.push_back([=](savsr_stream st) { return savsr_pack_frames(ctx, arena, x, t, h, w, dst_slot, st); });
  return 0;
}

extern "C" int savsr_plan_add_pack_frames_u8(savsr_plan* plan, savsr_arena* arena, const uint8_t* x, int t, int h, int w, int dst_slot) {
  SAVSR_REQUIRE(plan && arena && x, "savsr_plan_add_pack_frames_u8: null pointer");
  savsr_ctx* ctx = plan->ctx;
  plan->ops.push_back([=](savsr_stream st) { return savsr_pack_frames_u8(ctx, arena, x, t, h, w, dst_slot, st); });
  return 0;
}

extern "C" int savsr_plan_add_conv(savsr_plan* plan, savsr_arena* arena, const savsr_conv_group* groups, int ngroups, int ksize, int n_tile,
                                   int dst_mode, int impl) {
  SAVSR_REQUIRE(plan && arena && groups, "savsr_plan_add_conv: null pointer");
  SAVSR_REQUIRE(ngroups >= 0 && ngroups <= SAVSR_MAX_GROUPS, "savsr_plan_add_conv: ngroups %d out of range", ngroups);
  std::vector<savsr_conv_group> g(groups, groups + ngroups);
  savsr_ctx* ctx = plan->ctx;
  plan->ops.push_back([=](savsr_stream st) { return savsr_conv(ctx, arena, g.data(), ngroups, ksize, n_tile, dst_mode, impl, st); });
  return 0;
}

extern "C" int savsr_plan_add_osa_prologue(savsr_plan* plan, const savsr_osa_params* convs, int nconvs, int batch, int npart, int npix,
                                           float inv_scale_h, float inv_scale_w) {
  SAVSR_REQUIRE(plan && convs && nconvs >= 0, "savsr_plan_add_osa_prologue: null pointer");
  std::vector<savsr_osa_params> c(convs, convs + nconvs);
  savsr_ctx* ctx = plan->ctx;
  plan->ops.push_back([=](savsr_stream st) { return savsr_osa_prologue(ctx, c.data(), nconvs, batch, npart, npix, inv_scale_h, inv_scale_w, st); });
  return 0;
}

extern "C" int savsr_plan_add_ca_scale_residual(savsr_plan* plan, savsr_arena* arena, int t_slot, int x_slot, int dst_slot, const float* pool,
                                                int npart, const float* w1, const float* b1, const float* w2, const float* b2, float* y_scratch) {
  SAVSR_REQUIRE(plan && arena, "savsr_plan_add_ca_scale_residual: null pointer");
  savsr_ctx* ctx = plan->ctx;
  plan->ops.push_back([=](savsr_stream st) { return savsr_ca_scale_residual(ctx, arena, t_slot, x_slot, dst_slot, pool, npart, w1, b1, w2, b2, y_scratch, st); });
  return 0;
}

extern "C" int savsr_plan_add_osadapt_mask(savsr_plan* plan, const float* in16, int batch, int height, int width, const float* wa, const float* ba,
                                           const float* wb, const float* bb, const float* wc, const float* bc, float* half0, float* half1, float* mask) {
  SAVSR_REQUIRE(plan, "savsr_plan_add_osadapt_mask: null pointer");
  savsr_ctx* ctx = plan->ctx;
  plan->ops.push_back([=](savsr_stream st) { return savsr_osadapt_mask(ctx, in16, batch, height, width, wa, ba, wb, bb, wc, bc, half0, half1, mask, st); });
  return 0;
}

extern "C" int savsr_plan_add_satu_kconv_sta(savsr_plan* plan, savsr_arena* arena, int a_slot, int x_slot, int dst_slot, int h, int w,
                                             const void* weights, const float* bias, float slope) {
  SAVSR_REQUIRE(plan && arena, "savsr_plan_add_satu_kconv_sta: null pointer");
  savsr_ctx* ctx = plan->ctx;
  plan->ops.push_back([=](savsr_stream st) { return savsr_satu_kconv_sta(ctx, arena, a_slot, x_slot, dst_slot, h, w, weights, bias, slope, st); });
  return 0;
}

extern "C" int savsr_plan_add_satu_hr(savsr_plan* plan, savsr_arena* lr, int x_slot, int sta_slot, int h, int w, int H, int W, const float* table,
                                      const float* base_y, const float* base_x, const void* weights, const float* zbias, const float* tail_bias,
                                      const float* x_in, int t, int centre, float* out) {
  SAVSR_REQUIRE(plan && lr, "savsr_plan_add_satu_hr: null pointer");
  savsr_ctx* ctx = plan->ctx;
  plan->ops.push_back([=](savsr_stream st) {
    return savsr_satu_hr(ctx, lr, x_slot, sta_slot, h, w, H, W, table, base_y, base_x, weights, zbias, tail_bias, x_in, t, centre, out, st);
  });
  return 0;
}

extern "C" int savsr_plan_add_satu_hr_u8(savsr_plan* plan, savsr_arena* lr, int x_slot, int sta_slot, int h, int w, int H, int W,
                                         const float* table, const float* base_y, const float* base_x, const void* weights,
                                         const float* zbias, const float* tail_bias, const uint8_t* x_in, int t, int centre, uint8_t* out) {
  SAVSR_REQUIRE(plan && lr, "savsr_plan_add_satu_hr_u8: null pointer");
  savsr_ctx* ctx = plan->ctx;
  plan->ops.push_back([=](savsr_stream st) {
    return savsr_satu_hr_u8(ctx, lr, x_slot, sta_slot, h, w, H, W, table, base_y, base_x, weights, zbias, tail_bias, x_in, t, centre, out, st);
  });
  return 0;
}

extern "C" int savsr_plan_add_arena_export(savsr_plan* plan, savsr_arena* arena, int slot, float* nchw) {
  SAVSR_REQUIRE(plan && arena && nchw, "savsr_plan_add_arena_export: null pointer");
  plan->ops.push_back([=](savsr_stream st) { return savsr_arena_export(arena, slot, nchw, st); });
  return 0;
}

extern "C" int savsr_plan_run(savsr_plan* plan, savsr_stream st) {
  SAVSR_REQUIRE(plan, "savsr_plan_run: null plan");
  plan->ctx->fmt = plan->format;             // the operand format is context state read at launch
  for (size_t i = 0; i < plan->ops.size(); ++i) {
    const int rc = plan->ops[i](st);
    if (rc) return rc;                       // savsr_last_error() holds the failing launch's message
  }
  return 0;
}

static int forward(const char* name, savsr_plan* plan, const void* x, void* out, bool u8, savsr_stream st) {
  SAVSR_REQUIRE(plan && x && out, "%s: null pointer", name);
  SAVSR_REQUIRE(plan->x_in && plan->out, "%s: the plan has no I/O staging buffers (savsr_plan_set_io / savsr_plan_set_io_u8)", name);
  SAVSR_REQUIRE(plan->u8 == u8, "%s: the plan was set up for %s I/O; call %s", name, plan->u8 ? "uint8 BGR" : "fp32",
                plan->u8 ? "savsr_forward_u8" : "savsr_forward");
  DeviceGuard guard(plan->ctx->device);
  cudaStream_t s = static_cast<cudaStream_t>(st);
  if (x != plan->x_in) SAVSR_CUDA(cudaMemcpyAsync(plan->x_in, x, plan->x_bytes, cudaMemcpyDeviceToDevice, s));
  if (int rc = savsr_plan_run(plan, st)) return rc;
  if (out != plan->out) SAVSR_CUDA(cudaMemcpyAsync(out, plan->out, plan->out_bytes, cudaMemcpyDeviceToDevice, s));
  return 0;
}

extern "C" int savsr_forward(savsr_plan* plan, const float* x, float* out, savsr_stream st) {
  return forward("savsr_forward", plan, x, out, false, st);
}

extern "C" int savsr_forward_u8(savsr_plan* plan, const uint8_t* x, uint8_t* out, savsr_stream st) {
  return forward("savsr_forward_u8", plan, x, out, true, st);
}
