// extern "C" surface of libvr_b200.so; declarations and the reference call each entry replaces are in
// include/vr_b200.h.
#include <stdio.h>
#include <string.h>

#include <string>

#include "../../include/vr_b200.h"
#include "engine.h"
#include "kernels.h"
#include "tc_plan.h"

struct vr_ctx {
  vr::Engine* eng;
  std::string err;
};

static std::string g_create_err;

static int fail(vr_ctx* c, const std::string& m) {
  if (c) c->err = m;
  return -1;
}
static int done(vr_ctx* c, bool ok) {
  if (ok) return 0;
  c->err = c->eng->err;
  return -1;
}
#define CHECK_CTX(c) \
  if (!(c) || !(c)->eng) return -2;

extern "C" {

int vr_create(const vr_config* cfg, vr_ctx** out) {
  if (!cfg || !out) return -2;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    g_create_err = "no CUDA device visible: libvr_b200 has no CPU path";
    return -1;
  }
  if (cfg->device < 0 || cfg->device >= ndev) {
    g_create_err = "invalid device ordinal";
    return -1;
  }
  int nf = cfg->n_fft;
  if (nf < 64 || nf > 4096 || (nf & (nf - 1))) {
    g_create_err = "n_fft must be a power of two in [64, 4096]";
    return -1;
  }
  if (cfg->hop_length <= 0 || cfg->hop_length > nf) {
    g_create_err = "hop_length must be in (0, n_fft]";
    return -1;
  }
  if (cfg->max_batch <= 0 || cfg->cropsize <= 0) {
    g_create_err = "max_batch and cropsize must be positive";
    return -1;
  }
  vr::Config c;
  c.device = cfg->device; c.n_fft = cfg->n_fft; c.hop = cfg->hop_length; c.nout = cfg->nout;
  c.nout_lstm = cfg->nout_lstm; c.cropsize = cfg->cropsize; c.max_batch = cfg->max_batch;
  c.conv_mode = cfg->conv_mode;
  vr_ctx* ctx = new vr_ctx();
  ctx->eng = new vr::Engine(c);
  if (!ctx->eng->err.empty()) {
    g_create_err = ctx->eng->err;
    delete ctx->eng;
    delete ctx;
    return -1;
  }
  *out = ctx;
  return 0;
}

void vr_destroy(vr_ctx* ctx) {
  if (!ctx) return;
  delete ctx->eng;
  delete ctx;
}

const char* vr_last_error(const vr_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

int vr_load_tensor(vr_ctx* ctx, const char* name, int32_t dtype, int32_t ndim, const int64_t* shape,
                   const void* host_data) {
  CHECK_CTX(ctx);
  if (!name || (!host_data) || ndim < 0 || ndim > 8) return fail(ctx, "vr_load_tensor: bad arguments");
  return done(ctx, ctx->eng->load_tensor(name, dtype, ndim, shape, host_data));
}

int vr_finalize_weights(vr_ctx* ctx) {
  CHECK_CTX(ctx);
  return done(ctx, ctx->eng->finalize());
}

int vr_stft(vr_ctx* ctx, const float* wave, int64_t L, void* spec, int64_t T, float* absmax, void* stream) {
  CHECK_CTX(ctx);
  return done(ctx, ctx->eng->stft(wave, L, (float2*)spec, T, absmax, (cudaStream_t)stream));
}

int vr_istft(vr_ctx* ctx, const void* spec, int64_t T, float* wave, void* stream) {
  CHECK_CTX(ctx);
  return done(ctx, ctx->eng->istft((const float2*)spec, nullptr, T, wave, nullptr, (cudaStream_t)stream));
}

int vr_predict_mask(vr_ctx* ctx, const float* mag, int32_t N, float* mask, void* stream) {
  CHECK_CTX(ctx);
  return done(ctx, ctx->eng->predict_mask(mag, N, mask, ctx->eng->cfg().offset, (cudaStream_t)stream));
}

int vr_forward(vr_ctx* ctx, const float* mag, int32_t N, float* mask, void* stream) {
  CHECK_CTX(ctx);
  return done(ctx, ctx->eng->predict_mask(mag, N, mask, 0, (cudaStream_t)stream));
}

int vr_normaliser(vr_ctx* ctx, const void* spec, int64_t T, int32_t norm_mode, float* out, void* stream) {
  CHECK_CTX(ctx);
  return done(ctx, ctx->eng->normaliser((const float2*)spec, T, norm_mode, out, (cudaStream_t)stream));
}

int vr_separate_windows(vr_ctx* ctx, const void* spec, int64_t T, const float* norm, int32_t pad_l,
                        int32_t first_window, int32_t n_windows, float* mask, int64_t mask_T, int64_t frame_shift,
                        int32_t accumulate, void* stream) {
  CHECK_CTX(ctx);
  return done(ctx, ctx->eng->separate_windows((const float2*)spec, T, norm, pad_l, first_window, n_windows, mask,
                                              mask_T, frame_shift, accumulate, (cudaStream_t)stream));
}

int vr_separate(vr_ctx* ctx, const void* spec, int64_t T, int32_t tta, float* mask, void* stream) {
  CHECK_CTX(ctx);
  return done(ctx, ctx->eng->separate((const float2*)spec, T, tta, mask, (cudaStream_t)stream));
}

int vr_apply_mask(vr_ctx* ctx, const void* spec, const float* mask, int64_t T, void* y_spec, void* v_spec,
                  void* stream) {
  CHECK_CTX(ctx);
  return done(ctx, ctx->eng->apply_mask((const float2*)spec, mask, T, (float2*)y_spec, (float2*)v_spec,
                                        (cudaStream_t)stream));
}

int vr_mask_frame_min(vr_ctx* ctx, const float* mask, int64_t T, float* frame_min, void* stream) {
  CHECK_CTX(ctx);
  cudaSetDevice(ctx->eng->cfg().device);
  ++ctx->eng->launches;
  cudaError_t e = vr::launch_mask_frame_min(mask, 2 * ctx->eng->bins(), T, frame_min, (cudaStream_t)stream);
  return e == cudaSuccess ? 0 : fail(ctx, std::string("vr_mask_frame_min: ") + cudaGetErrorString(e));
}

int vr_mask_apply_weight(vr_ctx* ctx, float* mask, int64_t T, const float* weight, void* stream) {
  CHECK_CTX(ctx);
  cudaSetDevice(ctx->eng->cfg().device);
  ++ctx->eng->launches;
  cudaError_t e = vr::launch_mask_apply_weight(mask, 2 * ctx->eng->bins(), T, weight, (cudaStream_t)stream);
  return e == cudaSuccess ? 0 : fail(ctx, std::string("vr_mask_apply_weight: ") + cudaGetErrorString(e));
}

int vr_apply_mask_istft(vr_ctx* ctx, const void* spec, const float* mask, int64_t T, float* wave_inst,
                        float* wave_voc, void* stream) {
  CHECK_CTX(ctx);
  if (!mask) return fail(ctx, "vr_apply_mask_istft: mask is NULL");
  return done(ctx, ctx->eng->istft((const float2*)spec, mask, T, wave_inst, wave_voc, (cudaStream_t)stream));
}

int vr_stft_range(vr_ctx* ctx, const float* wave, int64_t L, void* spec, int64_t T, int64_t t0, int64_t t1,
                  void* stream) {
  CHECK_CTX(ctx);
  return done(ctx, ctx->eng->stft_range(wave, L, (float2*)spec, T, t0, t1, (cudaStream_t)stream));
}

int vr_normaliser_range(vr_ctx* ctx, const void* spec, int64_t T, int64_t t0, int64_t t1, float* out, void* stream) {
  CHECK_CTX(ctx);
  return done(ctx, ctx->eng->normaliser_range((const float2*)spec, T, t0, t1, out, (cudaStream_t)stream));
}

int vr_apply_mask_istft_range(vr_ctx* ctx, const void* spec, const float* mask, int64_t T, int64_t k0, int64_t k1,
                              float* wave_inst, float* wave_voc, void* stream) {
  CHECK_CTX(ctx);
  if (!mask) return fail(ctx, "vr_apply_mask_istft_range: mask is NULL");
  return done(ctx, ctx->eng->istft_range((const float2*)spec, mask, T, k0, k1, wave_inst, wave_voc,
                                         (cudaStream_t)stream));
}

int vr_separate_wave(vr_ctx* ctx, const float* wave, int64_t L, int32_t tta, float* wave_inst, float* wave_voc,
                     void* stream) {
  CHECK_CTX(ctx);
  return done(ctx, ctx->eng->separate_wave(wave, L, tta, wave_inst, wave_voc, (cudaStream_t)stream));
}

int vr_separate_wave_host(vr_ctx* ctx, const float* wave_host, int64_t L, int32_t tta, float* inst_host,
                          float* voc_host, void* stream) {
  CHECK_CTX(ctx);
  return done(ctx, ctx->eng->separate_wave_host(wave_host, L, tta, inst_host, voc_host, (cudaStream_t)stream));
}

int vr_separate_many(vr_ctx* ctx, int32_t n_tracks, const void* const* specs, const int64_t* T, int32_t tta,
                     float* const* masks, void* stream) {
  CHECK_CTX(ctx);
  // everything is checked before anything is launched
  if (n_tracks < 1) return fail(ctx, "vr_separate_many: n_tracks must be >= 1");
  if (!specs || !T || !masks) return fail(ctx, "vr_separate_many: specs, T and masks must not be NULL");
  for (int32_t i = 0; i < n_tracks; ++i) {
    const std::string at = "vr_separate_many: track " + std::to_string(i) + ": ";
    if (!specs[i]) return fail(ctx, at + "specs[i] is NULL");
    if (!masks[i]) return fail(ctx, at + "masks[i] is NULL");
    if (T[i] < 1) return fail(ctx, at + "T[i] must be >= 1");
  }
  return done(ctx, ctx->eng->separate_many((const float2* const*)specs, T, n_tracks, tta, masks, (cudaStream_t)stream));
}

int vr_separate_waves(vr_ctx* ctx, int32_t n_tracks, const float* const* waves, const int64_t* L, int32_t tta,
                      float* const* inst, float* const* voc, void* stream) {
  CHECK_CTX(ctx);
  if (n_tracks < 1) return fail(ctx, "vr_separate_waves: n_tracks must be >= 1");
  if (!waves || !L || !inst || !voc) return fail(ctx, "vr_separate_waves: waves, L, inst and voc must not be NULL");
  for (int32_t i = 0; i < n_tracks; ++i) {
    const std::string at = "vr_separate_waves: track " + std::to_string(i) + ": ";
    if (!waves[i]) return fail(ctx, at + "waves[i] is NULL");
    if (!inst[i]) return fail(ctx, at + "inst[i] is NULL");
    if (!voc[i]) return fail(ctx, at + "voc[i] is NULL");
    if (L[i] < 0) return fail(ctx, at + "L[i] must be >= 0");
  }
  return done(ctx, ctx->eng->separate_waves(waves, L, n_tracks, tta, inst, voc, (cudaStream_t)stream));
}

int vr_resample(vr_ctx* ctx, const float* x, int32_t channels, int64_t n_in, float* y, int64_t n_out, double sample_ratio,
                const double* win, const double* delta, int32_t nwin, int32_t table_per_crossing, void* stream) {
  // ctx may be NULL (audio is usually loaded before a model context exists): the call then runs on the calling
  // thread's current device and its error message is read with vr_last_error(NULL)
  auto bad = [&](const std::string& m) {
    if (ctx) return fail(ctx, m);
    g_create_err = m;
    return -1;
  };
  if (!x || !y || !win || !delta) return bad("vr_resample: null pointer");
  if (n_out != (int64_t)((double)n_in * sample_ratio))
    return bad("vr_resample: n_out must be int(n_in * sample_ratio) (resampy.core.resample)");
  if (ctx && ctx->eng) cudaSetDevice(ctx->eng->cfg().device);
  cudaError_t e = vr::launch_resample_sinc(x, channels, n_in, y, n_out, sample_ratio, win, delta, nwin, table_per_crossing,
                                           (cudaStream_t)stream);
  if (e != cudaSuccess) return bad(std::string("vr_resample: ") + cudaGetErrorString(e));
  return 0;
}

int vr_shared_alloc(vr_ctx* ctx, int64_t bytes, void** dev_ptr, unsigned char* handle64) {
  CHECK_CTX(ctx);
  if (!dev_ptr || !handle64 || bytes <= 0) return fail(ctx, "vr_shared_alloc: bad arguments");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle is 64 bytes");
  cudaSetDevice(ctx->eng->cfg().device);
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, (size_t)bytes);
  if (e != cudaSuccess) return fail(ctx, std::string("vr_shared_alloc: cudaMalloc: ") + cudaGetErrorString(e));
  cudaIpcMemHandle_t h;
  e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    return fail(ctx, std::string("vr_shared_alloc: cudaIpcGetMemHandle: ") + cudaGetErrorString(e));
  }
  memcpy(handle64, &h, 64);
  *dev_ptr = p;
  return 0;
}

int vr_shared_open(vr_ctx* ctx, const unsigned char* handle64, void** dev_ptr) {
  CHECK_CTX(ctx);
  if (!dev_ptr || !handle64) return fail(ctx, "vr_shared_open: bad arguments");
  cudaSetDevice(ctx->eng->cfg().device);
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  void* p = nullptr;
  cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) return fail(ctx, std::string("vr_shared_open: cudaIpcOpenMemHandle: ") + cudaGetErrorString(e));
  *dev_ptr = p;
  return 0;
}

int vr_shared_close(vr_ctx* ctx, void* dev_ptr, int32_t owner) {
  CHECK_CTX(ctx);
  if (!dev_ptr) return 0;
  cudaSetDevice(ctx->eng->cfg().device);
  cudaError_t e = owner ? cudaFree(dev_ptr) : cudaIpcCloseMemHandle(dev_ptr);
  if (e != cudaSuccess) return fail(ctx, std::string("vr_shared_close: ") + cudaGetErrorString(e));
  return 0;
}

int64_t vr_launch_count(const vr_ctx* ctx) { return ctx && ctx->eng ? ctx->eng->launches : 0; }

int vr_profile_enable(vr_ctx* ctx, int32_t on) {
  CHECK_CTX(ctx);
  ctx->eng->profile_enable(on != 0);
  return 0;
}

int vr_profile_read(vr_ctx* ctx, double* out6) {
  CHECK_CTX(ctx);
  return done(ctx, ctx->eng->profile_read(out6));
}

int vr_profile_dump(vr_ctx* ctx, char* text, int64_t cap, int64_t* needed) {
  CHECK_CTX(ctx);
  std::string t;
  if (!ctx->eng->profile_dump(t)) return done(ctx, false);
  if (needed) *needed = (int64_t)t.size() + 1;
  if (text && cap > 0) {
    const size_t n = t.size() < (size_t)cap - 1 ? t.size() : (size_t)cap - 1;
    memcpy(text, t.data(), n);
    text[n] = 0;
  }
  return 0;
}

int vr_debug_conv(vr_ctx* ctx, const float* x, int32_t N, int32_t Cin, int32_t H, int32_t W, const float* w,
                  const float* bias, int32_t Cout, int32_t k, int32_t stride, int32_t dil_h, int32_t dil_w, int32_t act,
                  int32_t use_tc, float* y, void* stream) {
  CHECK_CTX(ctx);
  return done(ctx, ctx->eng->debug_conv(x, N, Cin, H, W, w, bias, Cout, k, stride, dil_h, dil_w, act, use_tc, y,
                                        (cudaStream_t)stream));
}

int vr_debug_decoder(vr_ctx* ctx, const float* low, int32_t N, int32_t Cl, int32_t h, int32_t w, const float* skip,
                     int32_t Cs, const float* wgt, const float* bias, int32_t Cout, int32_t act, int32_t fused, float* y,
                     void* stream) {
  CHECK_CTX(ctx);
  return done(ctx, ctx->eng->debug_decoder(low, N, Cl, h, w, skip, Cs, wgt, bias, Cout, act, fused, y,
                                           (cudaStream_t)stream));
}

int vr_debug_set(int32_t key, int32_t value) {
  if (key < 0 || key >= 8) return -1;
  vr::g_tc_debug[key] = value;
  return 0;
}

int64_t vr_debug_trace(uint64_t* host_out, int64_t capacity) {
  return vr::tc_rows_read_trace((unsigned long long*)host_out, (long long)capacity);
}

int vr_debug_read(vr_ctx* ctx, const char* what, float* out, int64_t capacity, int64_t* dims, void* stream) {
  CHECK_CTX(ctx);
  return done(ctx, ctx->eng->debug_read(what, out, capacity, dims, (cudaStream_t)stream));
}

}  // extern "C"
