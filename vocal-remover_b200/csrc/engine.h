// Host-side engine: owns the device arena, the packed checkpoint and the per-layer launch plan of
// the CascadedNet forward (reference lib/nets.py:44-141) and the Separator glue (inference.py:16-102).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <functional>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "common.cuh"
#include "kernels.h"

namespace vr {

struct HostTensor {
  std::vector<int64_t> shape;
  std::vector<float> data;
};

struct Buffer {   // a whole NHWC split-bf16 allocation
  bf16* hi = nullptr;
  bf16* lo = nullptr;
  int N = 0, H = 0, W = 0, C = 0;
  int Wp = 0;   // row pitch in pixels (>= W): the Wp - W trailing pixels of every row are permanent zeros
  ActView view(int n, int h0, int h, int c0, int c) const {
    ActView v;
    const int64_t off = (int64_t)h0 * Wp * C + c0;
    v.hi = hi + off;
    v.lo = lo + off;
    v.N = n; v.H = h; v.W = W; v.C = c;
    v.sn = (int64_t)H * Wp * C;
    v.sh = (int64_t)Wp * C;
    v.sw = C;
    return v;
  }
  ActView all(int n) const { return view(n, 0, H, 0, C); }
};

struct TcConv;   // tcgen05 plan (conv_tc.cu)

struct ConvLayer {
  std::string name;
  int Cin = 0, CinPad = 0, Cout = 0, CoutPad = 0;
  int k = 1, stride = 1, dil_h = 1, dil_w = 1, act = ACT_RELU;
  float* w = nullptr;      // device fp32 [taps][CinPad][CoutPad]
  float* bias = nullptr;   // device fp32 [CoutPad]
  std::vector<float> w_host;     // packed copy kept for the tensor-core packer
  std::vector<float> bias_host;
  bool rows_wide = false;        // row kernel: 64 output channels per tile (decoder layers whose upsample is fused)
  // set around ONE launch by the caller: the row kernel also accumulates sum_c dot_w[c] * y[c] per output pixel into the
  // pre-zeroed plane dot_out[n][h][w] (the LSTM branch's 1x1 input convolution fused into dec2)
  const float* dot_w = nullptr;
  float* dot_out = nullptr;
  std::shared_ptr<TcConv> tc;    // null -> CUDA-core kernel
};

struct LstmPlan {
  int C = 0, bins = 0, hid = 0, T = 0;
  float* conv_w = nullptr;   // [C] folded
  float conv_bias = 0.f;
  float* wih = nullptr;      // [8*hid][bins]  (forward rows then reverse rows)
  float* bih = nullptr;      // [8*hid]        bias_ih + bias_hh
  float* whh = nullptr;      // [2][4*hid][hid]
  float* wd = nullptr;       // [bins][2*hid]
  float* dscale = nullptr;   // [bins]  BatchNorm1d scale
  float* dshift = nullptr;   // [bins]  scale*linear_bias + BatchNorm1d shift
  float* l0 = nullptr;       // [N][bins][T]  1x1 convolution, pre-activation
  float* xp = nullptr;       // [N][T][8*hid]
  float* hs = nullptr;       // [N][T][2*hid]
  float* y = nullptr;        // [bins][N][T]  the branch output at half resolution
};

struct BaseNetPlan {
  std::string prefix;
  int n = 0, H = 0, W = 0;
  ConvLayer enc1, enc_a[4], enc_b[4], aspp1, aspp2, aspp_d[3], bott, dec[4];   // dec[0]=dec4 .. dec[3]=dec1
  LstmPlan lstm;
  // skip_only: dec1's upsample of h is fused into the row kernel and d2 = [h 2n] only; the single LSTM channel is
  // up-sampled by a small kernel from lstm.y (half resolution, fp32 plane) into a 16-channel group at full
  // resolution: channels [n, n+16) of cat1 = [e1 n | up(lstm) 1 + 15 zeros] when e1 leaves room in its chunk (n = 16),
  // else an 8-channel group in the buffer lstm_up of its own (n = 32, 64: cat1 = [e1 n] stays dense for enc2.conv1, and
  // the row kernel reads the group as its last chunk through a second tensor map whose box TMA zero-fills).  Otherwise (CUDA-core validation mode, nets whose
  // 2n is not a multiple of 32): cat1 = [up(h) 2n | up(lstm) 1 + 15 zeros | e1 n | pad], d2 = [h 2n | lstm 1 | zeros].
  bool skip_only = false;
  int e1_coff = 0;          // channel offset of e1 inside cat1
  int lstm_coff = 0;        // skip_only: channel offset of the up-sampled LSTM channel inside cat1 (or 0 in lstm_up)
  bool lstm_own = false;    // skip_only: the up-sampled LSTM group lives in lstm_up, not in cat1
  Buffer cat1, t2, cat2, t3, cat3, t4, cat4, t5, e5, pool, f1, acat, ao, d4, d3, d2, lstm_up;
  int e1_off = 0;   // position of e1 in dec1's reduction (weight) order
};

struct Config {
  int device = 0;
  int n_fft = 2048, hop = 1024, nout = 32, nout_lstm = 128, cropsize = 256, max_batch = 4;
  int offset = 64;
  int conv_mode = 0;   // 0: tcgen05 where eligible, 1: CUDA-core kernel everywhere (validation)
};

class Engine {
 public:
  explicit Engine(const Config& cfg);
  ~Engine();

  std::string err;

  bool load_tensor(const char* name, int dtype, int ndim, const int64_t* shape, const void* data);
  bool finalize();
  bool ready() const { return finalized_; }

  // ---- reference-surface operations (device pointers) ----
  bool stft(const float* wave, int64_t L, float2* spec, int64_t T, float* absmax, cudaStream_t s);
  bool istft(const float2* spec, const float* mask, int64_t T, float* wave_a, float* wave_b, cudaStream_t s);
  bool stft_range(const float* wave, int64_t L, float2* spec, int64_t T, int64_t t0, int64_t t1, cudaStream_t s);
  bool normaliser_range(const float2* spec, int64_t T, int64_t t0, int64_t t1, float* out, cudaStream_t s);
  bool istft_range(const float2* spec, const float* mask, int64_t T, int64_t k0, int64_t k1, float* wave_a,
                   float* wave_b, cudaStream_t s);
  bool predict_mask(const float* mag, int N, float* mask_out, int offset, cudaStream_t s);
  // windows [first, first+count) of the padded spectrogram -> mask frames; see include/vr_b200.h
  bool separate_windows(const float2* spec, int64_t T, const float* norm, int pad_l, int first, int count,
                        float* mask, int64_t mask_T, int64_t frame_shift, int accumulate, cudaStream_t s,
                        bool final_pass = false);
  bool separate(const float2* spec, int64_t T, int tta, float* mask, cudaStream_t s);
  bool apply_mask(const float2* spec, const float* mask, int64_t T, float2* y, float2* v, cudaStream_t s);
  bool separate_wave(const float* wave, int64_t L, int tta, float* inst, float* voc, cudaStream_t s);
  bool separate_wave_host(const float* wave, int64_t L, int tta, float* inst, float* voc, cudaStream_t s);
  bool normaliser(const float2* spec, int64_t T, int mode, float* out, cudaStream_t s);
  // several tracks per call, their windows packed into shared forward batches (include/vr_b200.h vr_separate_many,
  // vr_separate_waves); arguments already validated
  bool separate_many(const float2* const* specs, const int64_t* T, int n, int tta, float* const* masks, cudaStream_t s);
  bool separate_waves(const float* const* waves, const int64_t* L, int n, int tta, float* const* inst,
                      float* const* voc, cudaStream_t s);

  // debug / tests: run one reference Conv2DBNActiv-shaped layer through a chosen kernel
  bool debug_conv(const float* x_nchw, int N, int Cin, int H, int W, const float* w, const float* bias, int Cout,
                  int k, int stride, int dil_h, int dil_w, int act, int use_tc, float* y_nchw, cudaStream_t s);
  bool debug_decoder(const float* low_nchw, int N, int Cl, int h, int w, const float* skip_nchw, int Cs, const float* wgt,
                     const float* bias, int Cout, int act, int fused, float* y_nchw, cudaStream_t s);
  // debug: copy an internal activation (by name) of the last forward to NCHW fp32
  bool debug_read(const char* what, float* out, int64_t cap, int64_t* dims, cudaStream_t s);

  const Config& cfg() const { return cfg_; }
  int bins() const { return cfg_.n_fft / 2 + 1; }
  int roi() const { int r = cfg_.cropsize - 2 * cfg_.offset; return r == 0 ? cfg_.cropsize : r; }
  int64_t launches = 0;   // kernels launched by this engine (bench 'gpu_launches')

  // optional CUDA-event timing of every convolution launch (bench.py roofline object)
  void profile_enable(bool on);
  // sums over the events recorded since enable: [0] tensor-core conv ms, [1] tensor-core conv algorithmic FLOPs,
  // [2] tensor-core launches, [3] CUDA-core conv ms, [4] CUDA-core conv FLOPs, [5] CUDA-core launches
  bool profile_read(double* out6);
  bool profile_dump(std::string& text);   // one line per profiled launch: name N H W tc ms gflop

 private:
  Config cfg_;
  bool finalized_ = false;
  bool warned_simt_ = false;   // the CUDA-core fallback warning was printed
  std::map<std::string, HostTensor> sd_;
  std::vector<void*> allocs_;
  int last_n_ = 0;
  // tc: 1 = tensor-core convolution, 0 = CUDA-core convolution, 2 = any other kernel of the path
  struct ProfRec { cudaEvent_t a, b; double flops; int tc; std::string name; int N, H, W; };
  bool profiling_ = false;
  std::vector<ProfRec> prof_;
  int prof_begin(const std::string& name, int kind, double flops, int N, int H, int W, cudaStream_t s);
  void prof_end(int idx, cudaStream_t s);
  // a non-convolution launch, bracketed by a CUDA-event pair while profiling is on
  template <class F>
  bool timed(const char* name, int N, int H, int W, cudaStream_t s, F&& launch) {
    const int i = prof_begin(name, 2, 0.0, N, H, W, s);
    const bool ok = launch();
    prof_end(i, s);
    return ok;
  }

  // whole-track workspace (grow-only)
  float2* ws_spec_ = nullptr; int64_t ws_spec_cap_ = 0;
  float* ws_mask_ = nullptr; int64_t ws_mask_cap_ = 0;
  float* ws_frames_ = nullptr; int64_t ws_frames_cap_ = 0;
  float* ws_wave_ = nullptr; int64_t ws_wave_cap_ = 0;   // [2][L] in + 2 x [2][Lo] out (host-buffer entry)
  float* ws_norm_ = nullptr;            // [4] floats: absmax, lexmax-abs
  unsigned long long* ws_lex_ = nullptr;
  // several-track calls: one normaliser (and lexmax scratch) per track, grow-only
  float* ws_norms_ = nullptr; unsigned long long* ws_lexs_ = nullptr; int64_t ws_norms_cap_ = 0;

  // The tables of a several-track call (window descriptors, track tables) are built on the host, staged in a pinned
  // buffer and copied to the device once per call, on the call's stream.  The next call may rewrite the pinned buffer
  // only after that copy has run (ev_tab_copied_, waited on by the host), and the device table only after the previous
  // call's last reader (ev_tab_used_, waited on by the stream).
  struct Tables {
    std::vector<unsigned char> bytes;
    template <class X>
    size_t put(const std::vector<X>& v) {
      const size_t off = (bytes.size() + 15) / 16 * 16;
      bytes.resize(off + sizeof(X) * v.size());
      if (!v.empty()) memcpy(bytes.data() + off, v.data(), sizeof(X) * v.size());
      return off;
    }
  };
  unsigned char* tab_host_ = nullptr; size_t tab_host_cap_ = 0;
  unsigned char* tab_dev_ = nullptr; size_t tab_dev_cap_ = 0;
  cudaEvent_t ev_tab_copied_ = nullptr, ev_tab_used_ = nullptr;
  bool upload_tables(const Tables& t, cudaStream_t s, const unsigned char** dev);
  // flat window schedule of a several-track call, cut into forward batches: batch b is wins[chunk_end[b-1], chunk_end[b])
  struct Schedule {
    std::vector<WinDesc> wins;
    std::vector<int> chunk_end;
  };
  void schedule_windows(const float2* const* specs, const int64_t* T, int n, int tta, float* const* masks,
                        Schedule& sch) const;
  bool run_schedule(const Schedule& sch, const WinDesc* d_wins, cudaStream_t s);
  bool normalisers_many(const NormTrack* d_tracks, int n, int64_t max_n, int mode, cudaStream_t s);
  bool ensure_norms(int n);

  // the high-band BaseNets of stages 1-2 run on their own stream next to the low-band chain (independent until
  // stage 3, lib/nets.py:88-99); disabled while per-kernel profiling is on so event timings stay per-kernel
  cudaStream_t s_hi_ = nullptr;
  // host-buffer entry: finished output spans are copied back on their own stream while the next window batch computes
  cudaStream_t s_copy_ = nullptr;
  cudaEvent_t ev_span_ = nullptr;
  std::function<bool(int64_t)> on_frames_final_;   // called after a batch of the last pass: mask frames [0, f) are final
  cudaEvent_t ev_fork_ = nullptr, ev_join_ = nullptr, ev_lstm_fork_ = nullptr, ev_lstm_join_ = nullptr;

  float2* twiddle_ = nullptr;
  float* window_ = nullptr;

  Buffer in3_;                 // (Nb, max_bin, W, C3): [aux2 | aux1 | x | pad]
  int pos_aux2_ = 0, pos_aux1_ = 0, pos_x_ = 0;
  Buffer o1_, o2_;             // low-band BaseNet outputs before the 1x1 bridge (stage 1 / stage 2)
  Buffer f3_;                  // stage-3 output (Nb, max_bin, W, nout)
  BaseNetPlan nets_[5];        // stg1_low, stg1_high, stg2_low, stg2_high, stg3_full
  ConvLayer bridge1_, bridge2_;
  float* out_w_ = nullptr;     // [2][nout]

  void* dalloc(size_t bytes);
  Buffer make_buffer(int N, int H, int W, int C, int pad_w = 0);
  bool need(const std::string& key, std::initializer_list<int64_t> shape, const HostTensor** out);
  bool make_conv(ConvLayer& L, const std::string& prefix, const std::vector<int>& perm, int cin_pad, int k, int stride,
                 int dh, int dw, int act);
  bool build_basenet(BaseNetPlan& P, const std::string& prefix, int nin, const std::vector<int>& in_perm, int cin_pad,
                     int n, int H, int W, int nin_lstm, int nout_lstm);
  bool run_conv(ConvLayer& L, const ActView& in, const ActView& out, cudaStream_t s, const ActView* up_src = nullptr,
                const ActView* extra = nullptr);
  bool run_conv_inner(ConvLayer& L, const ActView& in, const ActView& out, bool use_tc, cudaStream_t s,
                      const ActView* up_src, const ActView* extra);
  // Decoder (lib/layers.py:51-64): upsample `low` into channels [0, low.C) of `cat`, then conv(cat) -> out; the
  // upsample is fused into the convolution's operand producer when the row kernel can do it
  bool run_decoder(ConvLayer& L, const ActView& low, const Buffer& cat, int N, const ActView& out, cudaStream_t s);
  bool run_basenet(BaseNetPlan& P, const ActView& in, const ActView& out, int N, cudaStream_t s,
                   cudaStream_t side = nullptr);
  bool forward(int N, cudaStream_t s);   // in3_ x-channels already packed for N windows -> f3_
  bool ensure_ws(int64_t T);
  bool ck(cudaError_t e, const char* what);
};

// conv_tc.cu
bool tc_supported(const ConvLayer& L, const ActView& in, const ActView& out);
bool tc_prepare(ConvLayer& L, std::string& err, std::vector<void*>& allocs);
cudaError_t tc_launch(ConvLayer& L, const ActView& in, const ActView& out, cudaStream_t s, std::string& err,
                      const ActView* up_src = nullptr, const ActView* extra = nullptr);
bool tc_can_fuse_upsample(const ConvLayer& L, const ActView& in, const ActView& out, const ActView& up_src);

}  // namespace vr
