// Engine: checkpoint packing, device arena and the launch sequence of the hot path.
// Reference call stack being replaced: inference.py:70-102 (Separator.separate / separate_tta) ->
// inference.py:42-68 (_separate) -> lib/nets.py:124-131 (predict_mask) -> lib/nets.py:82-117 (forward)
// -> lib/nets.py:26-41 (BaseNet) -> lib/layers.py.
#include "engine.h"
#include "tc_plan.h"

#include <math.h>
#include <stdio.h>
#include <string.h>

namespace vr {

static const double kBnEps = 1e-5;   // nn.BatchNorm2d / BatchNorm1d default eps

bool Engine::ck(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return true;
  err = std::string(what) + ": " + cudaGetErrorString(e);
  return false;
}

void* Engine::dalloc(size_t bytes) {
  void* p = nullptr;
  if (bytes == 0) bytes = 16;
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) {
    err = std::string("cudaMalloc(") + std::to_string(bytes) + "): " + cudaGetErrorString(e);
    return nullptr;
  }
  cudaMemset(p, 0, bytes);   // pad channels must be finite zeros forever (zero weights multiply them)
  allocs_.push_back(p);
  return p;
}

Buffer Engine::make_buffer(int N, int H, int W, int C, int pad_w) {
  Buffer b;
  b.N = N; b.H = H; b.W = W; b.C = C;
  b.Wp = W + pad_w;
  size_t plane = (size_t)N * H * b.Wp * C * sizeof(bf16);
  plane = (plane + 1023) / 1024 * 1024;
  char* p = (char*)dalloc(2 * plane);
  if (p) {
    b.hi = (bf16*)p;
    b.lo = (bf16*)(p + plane);
  }
  return b;
}

Engine::Engine(const Config& cfg) : cfg_(cfg) {
  if (cudaSetDevice(cfg_.device) != cudaSuccess) {
    err = "cudaSetDevice failed (no CUDA device? this library has no CPU path)";
    return;
  }
  const int NF = cfg_.n_fft;
  std::vector<float2> tw(NF / 2);
  std::vector<float> win(NF);
  for (int q = 0; q < NF / 2; ++q) {
    double a = -2.0 * M_PI * (double)q / (double)NF;
    tw[q] = make_float2((float)cos(a), (float)sin(a));
  }
  for (int n = 0; n < NF; ++n) win[n] = (float)(0.5 - 0.5 * cos(2.0 * M_PI * (double)n / (double)NF));
  twiddle_ = (float2*)dalloc(sizeof(float2) * tw.size());
  window_ = (float*)dalloc(sizeof(float) * win.size());
  ws_norm_ = (float*)dalloc(sizeof(float) * 4);
  ws_lex_ = (unsigned long long*)dalloc(sizeof(unsigned long long));
  if (!twiddle_ || !window_ || !ws_norm_ || !ws_lex_) return;
  cudaMemcpy(twiddle_, tw.data(), sizeof(float2) * tw.size(), cudaMemcpyHostToDevice);
  cudaMemcpy(window_, win.data(), sizeof(float) * win.size(), cudaMemcpyHostToDevice);
  cudaStreamCreateWithFlags(&s_hi_, cudaStreamNonBlocking);
  cudaStreamCreateWithFlags(&s_copy_, cudaStreamNonBlocking);
  cudaEventCreateWithFlags(&ev_span_, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&ev_fork_, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&ev_join_, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&ev_lstm_fork_, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&ev_lstm_join_, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&ev_tab_copied_, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&ev_tab_used_, cudaEventDisableTiming);
}

Engine::~Engine() {
  cudaSetDevice(cfg_.device);
  for (void* p : allocs_) cudaFree(p);
  if (ws_spec_) cudaFree(ws_spec_);
  if (ws_mask_) cudaFree(ws_mask_);
  if (ws_frames_) cudaFree(ws_frames_);
  if (ws_wave_) cudaFree(ws_wave_);
  if (ws_norms_) cudaFree(ws_norms_);
  if (ws_lexs_) cudaFree(ws_lexs_);
  if (tab_dev_) cudaFree(tab_dev_);
  if (tab_host_) cudaFreeHost(tab_host_);
  profile_enable(false);
  if (s_hi_) cudaStreamDestroy(s_hi_);
  if (s_copy_) cudaStreamDestroy(s_copy_);
  if (ev_span_) cudaEventDestroy(ev_span_);
  if (ev_fork_) cudaEventDestroy(ev_fork_);
  if (ev_join_) cudaEventDestroy(ev_join_);
  if (ev_lstm_fork_) cudaEventDestroy(ev_lstm_fork_);
  if (ev_lstm_join_) cudaEventDestroy(ev_lstm_join_);
  if (ev_tab_copied_) cudaEventDestroy(ev_tab_copied_);
  if (ev_tab_used_) cudaEventDestroy(ev_tab_used_);
}

bool Engine::load_tensor(const char* name, int dtype, int ndim, const int64_t* shape, const void* data) {
  HostTensor t;
  int64_t n = 1;
  for (int i = 0; i < ndim; ++i) {
    t.shape.push_back(shape[i]);
    n *= shape[i];
  }
  t.data.resize((size_t)n);
  if (dtype == 0) {
    memcpy(t.data.data(), data, sizeof(float) * (size_t)n);
  } else if (dtype == 1) {   // int64 (BatchNorm num_batches_tracked): kept only for strict key checking
    const int64_t* p = (const int64_t*)data;
    for (int64_t i = 0; i < n; ++i) t.data[(size_t)i] = (float)p[i];
  } else {
    err = std::string("unsupported dtype for tensor ") + name;
    return false;
  }
  sd_[name] = std::move(t);
  finalized_ = false;
  return true;
}

bool Engine::need(const std::string& key, std::initializer_list<int64_t> shape, const HostTensor** out) {
  auto it = sd_.find(key);
  if (it == sd_.end()) {
    err = "missing key in state_dict: " + key;
    return false;
  }
  std::vector<int64_t> s(shape);
  if (it->second.shape != s) {
    std::string got, want;
    for (auto d : it->second.shape) got += std::to_string(d) + ",";
    for (auto d : s) want += std::to_string(d) + ",";
    err = "size mismatch for " + key + ": checkpoint (" + got + ") vs model (" + want + ")";
    return false;
  }
  *out = &it->second;
  return true;
}

// Fold BatchNorm2d(eval) into the bias-free conv and pack to [tap][CinPad][CoutPad] (lib/layers.py:12-23).
// perm[packed_ci] = original input channel, or -1 for a zero (padding) channel.
bool Engine::make_conv(ConvLayer& L, const std::string& prefix, const std::vector<int>& perm, int cin_pad, int k,
                       int stride, int dh, int dw, int act) {
  L.name = prefix;
  L.k = k; L.stride = stride; L.dil_h = dh; L.dil_w = dw; L.act = act;
  auto itw = sd_.find(prefix + ".conv.0.weight");
  if (itw == sd_.end()) {
    err = "missing key in state_dict: " + prefix + ".conv.0.weight";
    return false;
  }
  const HostTensor& w = itw->second;
  if (w.shape.size() != 4 || w.shape[2] != k || w.shape[3] != k) {
    err = "size mismatch for " + prefix + ".conv.0.weight";
    return false;
  }
  const int Cout = (int)w.shape[0], Cin = (int)w.shape[1];
  int used = 0;
  for (int v : perm) used += v >= 0;
  if (used != Cin || (int)perm.size() != cin_pad) {
    err = "internal: channel permutation does not cover the input channels of " + prefix;
    return false;
  }
  const HostTensor *g, *b, *m, *v, *cnt;
  if (!need(prefix + ".conv.1.weight", {Cout}, &g) || !need(prefix + ".conv.1.bias", {Cout}, &b) ||
      !need(prefix + ".conv.1.running_mean", {Cout}, &m) || !need(prefix + ".conv.1.running_var", {Cout}, &v) ||
      !need(prefix + ".conv.1.num_batches_tracked", {}, &cnt))
    return false;
  L.Cin = Cin; L.CinPad = cin_pad; L.Cout = Cout; L.CoutPad = round_up(Cout, 8);
  const int taps = k * k;
  L.w_host.assign((size_t)taps * L.CinPad * L.CoutPad, 0.f);
  L.bias_host.assign((size_t)L.CoutPad, 0.f);
  for (int co = 0; co < Cout; ++co) {
    const double scale = (double)g->data[co] / sqrt((double)v->data[co] + kBnEps);
    L.bias_host[co] = (float)((double)b->data[co] - (double)m->data[co] * scale);
    for (int pc = 0; pc < cin_pad; ++pc) {
      const int ci = perm[pc];
      if (ci < 0) continue;
      for (int t = 0; t < taps; ++t)
        L.w_host[((size_t)t * L.CinPad + pc) * L.CoutPad + co] =
            (float)((double)w.data[((size_t)co * Cin + ci) * taps + t] * scale);
    }
  }
  L.w = (float*)dalloc(L.w_host.size() * sizeof(float));
  L.bias = (float*)dalloc(L.bias_host.size() * sizeof(float));
  if (!L.w || !L.bias) return false;
  cudaMemcpy(L.w, L.w_host.data(), L.w_host.size() * sizeof(float), cudaMemcpyHostToDevice);
  cudaMemcpy(L.bias, L.bias_host.data(), L.bias_host.size() * sizeof(float), cudaMemcpyHostToDevice);
  if (cfg_.conv_mode == 0) {
    if (!tc_prepare(L, err, allocs_)) return false;
  }
  return true;
}

static std::vector<int> identity_perm(int c, int pad) {
  std::vector<int> p((size_t)pad, -1);
  for (int i = 0; i < c; ++i) p[(size_t)i] = i;
  return p;
}

bool Engine::build_basenet(BaseNetPlan& P, const std::string& prefix, int nin, const std::vector<int>& in_perm,
                           int cin_pad, int n, int H, int W, int nin_lstm, int nout_lstm) {
  (void)nin;
  P.prefix = prefix; P.n = n; P.H = H; P.W = W;
  const int Nb = cfg_.max_batch;
  if (H % 16 || W % 16 || n % 4) {
    err = "unsupported geometry: band height and cropsize must be multiples of 16 and nout a multiple of 16";
    return false;
  }
  // Layouts of the dec1 input (see BaseNetPlan::skip_only in engine.h).  The fused layout needs the row kernel with
  // dec1's up-sampled half (h, 2n channels) in whole 32-channel chunks.
  P.skip_only = cfg_.conv_mode == 0 && g_tc_debug[5] == 1 && g_tc_debug[1] == 0 &&
                (2 * n) % 32 == 0 && W % 128 == 0 && H % 8 == 0;
  const int lg = 16;   // the lstm channel + 15 zeros keep every slice 32-byte aligned (full-sector 256-bit stores)
  P.lstm_own = P.skip_only && n % 32 == 0;
  const int c1 = P.skip_only ? 2 * n + round_up(n, 32) + (P.lstm_own ? lg : 0) : round_up(3 * n + lg, 16);
  P.e1_off = P.skip_only ? 2 * n : 2 * n + lg;      // position of e1 in dec1's reduction (weight) order
  P.e1_coff = P.skip_only ? 0 : P.e1_off;           // position of e1 in the cat1 buffer
  P.lstm_coff = !P.skip_only ? 2 * n : P.lstm_own ? 0 : n;
  P.cat1 = make_buffer(Nb, H, W, !P.skip_only ? c1 : P.lstm_own ? n : round_up(n + lg, 32));
  if (P.lstm_own) P.lstm_up = make_buffer(Nb, H, W, 8);   // 8-channel group: the row kernel's TMA box zero-fills the rest
  P.t2 = make_buffer(Nb, H / 2, W / 2, 2 * n);
  P.cat2 = make_buffer(Nb, H / 2, W / 2, 6 * n);
  P.t3 = make_buffer(Nb, H / 4, W / 4, 4 * n);
  P.cat3 = make_buffer(Nb, H / 4, W / 4, 10 * n);
  P.t4 = make_buffer(Nb, H / 8, W / 8, 6 * n);
  P.cat4 = make_buffer(Nb, H / 8, W / 8, 14 * n);
  P.t5 = make_buffer(Nb, H / 16, W / 16, 8 * n);
  P.e5 = make_buffer(Nb, H / 16, W / 16, 8 * n);
  P.pool = make_buffer(Nb, 1, W / 16, 8 * n);
  P.f1 = make_buffer(Nb, 1, W / 16, 8 * n);
  P.acat = make_buffer(Nb, H / 16, W / 16, 40 * n);
  P.ao = make_buffer(Nb, H / 16, W / 16, 8 * n);
  P.d4 = make_buffer(Nb, H / 8, W / 8, 6 * n);
  P.d3 = make_buffer(Nb, H / 4, W / 4, 4 * n);
  P.d2 = make_buffer(Nb, H / 2, W / 2, P.skip_only ? 2 * n : 2 * n + lg);
  if (!P.d2.hi || !P.cat1.hi) return false;

  if (!make_conv(P.enc1, prefix + ".enc1", in_perm, cin_pad, 3, 1, 1, 1, ACT_RELU)) return false;
  const int mult[5] = {1, 2, 4, 6, 8};
  for (int i = 0; i < 4; ++i) {
    const int cin = n * mult[i], cout = n * mult[i + 1];
    const std::string e = prefix + ".enc" + std::to_string(i + 2);
    if (!make_conv(P.enc_a[i], e + ".conv1", identity_perm(cin, round_up(cin, 8)), round_up(cin, 8), 3, 2, 1, 1,
                   ACT_LEAKY))
      return false;
    if (!make_conv(P.enc_b[i], e + ".conv2", identity_perm(cout, cout), cout, 3, 1, 1, 1, ACT_LEAKY)) return false;
  }
  const int c8 = 8 * n;
  if (!make_conv(P.aspp1, prefix + ".aspp.conv1.1", identity_perm(c8, c8), c8, 1, 1, 1, 1, ACT_RELU)) return false;
  if (!make_conv(P.aspp2, prefix + ".aspp.conv2", identity_perm(c8, c8), c8, 1, 1, 1, 1, ACT_RELU)) return false;
  const int dil[3][2] = {{4, 2}, {8, 4}, {12, 6}};   // lib/nets.py:10
  for (int i = 0; i < 3; ++i)
    if (!make_conv(P.aspp_d[i], prefix + ".aspp.conv" + std::to_string(i + 3), identity_perm(c8, c8), c8, 3, 1,
                   dil[i][0], dil[i][1], ACT_RELU))
      return false;
  if (!make_conv(P.bott, prefix + ".aspp.bottleneck", identity_perm(5 * c8, 5 * c8), 5 * c8, 1, 1, 1, 1, ACT_RELU))
    return false;
  if (!make_conv(P.dec[0], prefix + ".dec4.conv1", identity_perm(14 * n, 14 * n), 14 * n, 3, 1, 1, 1, ACT_RELU))
    return false;
  if (!make_conv(P.dec[1], prefix + ".dec3.conv1", identity_perm(10 * n, 10 * n), 10 * n, 3, 1, 1, 1, ACT_RELU))
    return false;
  P.dec[2].rows_wide = true;   // dec2's upsample is fused into the row kernel whenever 4n is a multiple of 32
  if (!make_conv(P.dec[2], prefix + ".dec2.conv1", identity_perm(6 * n, 6 * n), 6 * n, 3, 1, 1, 1, ACT_RELU))
    return false;
  {
    // dec1 input in the reference: cat[ up(cat[h (2n), lstm (1)]) , e1 (n) ]  (lib/nets.py:38-39, layers.py:52-56)
    // packed as [ up(h) 2n | up(lstm) 1 | 15 zeros | e1 n | zeros ], or (skip_only) [ up(h) 2n | e1 n | up(lstm) 1 | zeros ]
    std::vector<int> perm((size_t)c1, -1);
    for (int i = 0; i < 2 * n; ++i) perm[(size_t)i] = i;
    perm[(size_t)(!P.skip_only ? 2 * n : P.lstm_own ? 2 * n + round_up(n, 32) : 2 * n + n)] = 2 * n;
    for (int i = 0; i < n; ++i) perm[(size_t)(P.e1_off + i)] = 2 * n + 1 + i;
    // (the 64-wide tile was measured on dec1 as well - one N tile instead of two for n = 64 - and is no faster there:
    //  with its single accumulator set the epilogue no longer overlaps the next tile's products)
    if (!make_conv(P.dec[3], prefix + ".dec1.conv1", perm, c1, 3, 1, 1, 1, ACT_RELU)) return false;
  }

  // ---- LSTM module (lib/layers.py:110-122) ----
  LstmPlan& Q = P.lstm;
  const std::string lp = prefix + ".lstm_dec2";
  Q.C = 2 * n; Q.bins = H / 2; Q.T = W / 2; Q.hid = nout_lstm / 2;
  if (Q.bins != nin_lstm) {
    err = "LSTM input size does not match band height / 2 for " + lp;
    return false;
  }
  const HostTensor *cw, *g, *b, *m, *v, *cnt;
  if (!need(lp + ".conv.conv.0.weight", {1, Q.C, 1, 1}, &cw) || !need(lp + ".conv.conv.1.weight", {1}, &g) ||
      !need(lp + ".conv.conv.1.bias", {1}, &b) || !need(lp + ".conv.conv.1.running_mean", {1}, &m) ||
      !need(lp + ".conv.conv.1.running_var", {1}, &v) || !need(lp + ".conv.conv.1.num_batches_tracked", {}, &cnt))
    return false;
  {
    const double scale = (double)g->data[0] / sqrt((double)v->data[0] + kBnEps);
    std::vector<float> w((size_t)Q.C);
    for (int c = 0; c < Q.C; ++c) w[(size_t)c] = (float)((double)cw->data[(size_t)c] * scale);
    Q.conv_bias = (float)((double)b->data[0] - (double)m->data[0] * scale);
    Q.conv_w = (float*)dalloc(sizeof(float) * w.size());
    if (!Q.conv_w) return false;
    cudaMemcpy(Q.conv_w, w.data(), sizeof(float) * w.size(), cudaMemcpyHostToDevice);
  }
  {
    const int H4 = 4 * Q.hid;
    std::vector<float> wih((size_t)2 * H4 * Q.bins), bih((size_t)2 * H4), whh((size_t)2 * H4 * Q.hid);
    const char* sfx[2] = {"", "_reverse"};
    for (int d = 0; d < 2; ++d) {
      const HostTensor *a, *h, *b1, *b2;
      if (!need(lp + ".lstm.weight_ih_l0" + sfx[d], {H4, Q.bins}, &a) ||
          !need(lp + ".lstm.weight_hh_l0" + sfx[d], {H4, Q.hid}, &h) ||
          !need(lp + ".lstm.bias_ih_l0" + sfx[d], {H4}, &b1) || !need(lp + ".lstm.bias_hh_l0" + sfx[d], {H4}, &b2))
        return false;
      memcpy(&wih[(size_t)d * H4 * Q.bins], a->data.data(), sizeof(float) * (size_t)H4 * Q.bins);
      memcpy(&whh[(size_t)d * H4 * Q.hid], h->data.data(), sizeof(float) * (size_t)H4 * Q.hid);
      for (int i = 0; i < H4; ++i) bih[(size_t)d * H4 + i] = b1->data[(size_t)i] + b2->data[(size_t)i];
    }
    Q.wih = (float*)dalloc(sizeof(float) * wih.size());
    Q.bih = (float*)dalloc(sizeof(float) * bih.size());
    Q.whh = (float*)dalloc(sizeof(float) * whh.size());
    if (!Q.wih || !Q.bih || !Q.whh) return false;
    cudaMemcpy(Q.wih, wih.data(), sizeof(float) * wih.size(), cudaMemcpyHostToDevice);
    cudaMemcpy(Q.bih, bih.data(), sizeof(float) * bih.size(), cudaMemcpyHostToDevice);
    cudaMemcpy(Q.whh, whh.data(), sizeof(float) * whh.size(), cudaMemcpyHostToDevice);
  }
  {
    const int K = 2 * Q.hid;
    const HostTensor *dw, *db, *g1, *b1, *m1, *v1, *c1t;
    if (!need(lp + ".dense.0.weight", {Q.bins, K}, &dw) || !need(lp + ".dense.0.bias", {Q.bins}, &db) ||
        !need(lp + ".dense.1.weight", {Q.bins}, &g1) || !need(lp + ".dense.1.bias", {Q.bins}, &b1) ||
        !need(lp + ".dense.1.running_mean", {Q.bins}, &m1) || !need(lp + ".dense.1.running_var", {Q.bins}, &v1) ||
        !need(lp + ".dense.1.num_batches_tracked", {}, &c1t))
      return false;
    std::vector<float> sc((size_t)Q.bins), sh((size_t)Q.bins);
    for (int bin = 0; bin < Q.bins; ++bin) {
      const double s = (double)g1->data[(size_t)bin] / sqrt((double)v1->data[(size_t)bin] + kBnEps);
      sc[(size_t)bin] = (float)s;
      sh[(size_t)bin] = (float)(s * ((double)db->data[(size_t)bin] - (double)m1->data[(size_t)bin]) +
                                (double)b1->data[(size_t)bin]);
    }
    Q.wd = (float*)dalloc(sizeof(float) * dw->data.size());
    Q.dscale = (float*)dalloc(sizeof(float) * sc.size());
    Q.dshift = (float*)dalloc(sizeof(float) * sh.size());
    if (!Q.wd || !Q.dscale || !Q.dshift) return false;
    cudaMemcpy(Q.wd, dw->data.data(), sizeof(float) * dw->data.size(), cudaMemcpyHostToDevice);
    cudaMemcpy(Q.dscale, sc.data(), sizeof(float) * sc.size(), cudaMemcpyHostToDevice);
    cudaMemcpy(Q.dshift, sh.data(), sizeof(float) * sh.size(), cudaMemcpyHostToDevice);
  }
  Q.l0 = (float*)dalloc(sizeof(float) * (size_t)Nb * Q.T * Q.bins);
  Q.xp = (float*)dalloc(sizeof(float) * (size_t)Nb * Q.T * 8 * Q.hid);
  Q.hs = (float*)dalloc(sizeof(float) * (size_t)Nb * Q.T * 2 * Q.hid);
  Q.y = (float*)dalloc(sizeof(float) * (size_t)Nb * Q.T * Q.bins);
  return Q.l0 && Q.xp && Q.hs && Q.y;
}

bool Engine::finalize() {
  if (finalized_) return true;
  if (!err.empty() && !twiddle_) return false;
  cudaSetDevice(cfg_.device);
  const int max_bin = cfg_.n_fft / 2, W = cfg_.cropsize, Nb = cfg_.max_batch;
  const int nout = cfg_.nout, a1 = nout / 4, a2 = nout / 2;
  if (nout % 16) {
    err = "nout must be a multiple of 16";
    return false;
  }
  if (W - 2 * cfg_.offset <= 0) {   // lib/nets.py:129 assert
    err = "cropsize must be larger than 2*offset (AssertionError in the reference, lib/nets.py:129)";
    return false;
  }
  pos_aux2_ = 0; pos_aux1_ = a2; pos_x_ = a2 + a1;
  const int C3 = round_up(a2 + a1 + 2, 16);
  in3_ = make_buffer(Nb, max_bin, W, C3);
  o1_ = make_buffer(Nb, max_bin / 2, W, nout / 2);
  o2_ = make_buffer(Nb, max_bin / 2, W, nout);
  f3_ = make_buffer(Nb, max_bin, W, nout);
  if (!in3_.hi || !o1_.hi || !o2_.hi || !f3_.hi) return false;

  const int nin_lstm = max_bin / 2;
  // stage 1: input = [x]                      (lib/nets.py:59-65, 88-92)
  const int c0_1 = pos_x_ / 16 * 16, cp1 = round_up(pos_x_ + 2 - c0_1, 16);
  std::vector<int> p1((size_t)cp1, -1);
  p1[(size_t)(pos_x_ - c0_1)] = 0; p1[(size_t)(pos_x_ - c0_1 + 1)] = 1;
  // stage 2: input = cat[x, aux1]             (lib/nets.py:67-73, 95-98)
  const int c0_2 = pos_aux1_ / 16 * 16, cp2 = round_up(pos_x_ + 2 - c0_2, 16);
  std::vector<int> p2((size_t)cp2, -1);
  p2[(size_t)(pos_x_ - c0_2)] = 0; p2[(size_t)(pos_x_ - c0_2 + 1)] = 1;
  for (int j = 0; j < a1; ++j) p2[(size_t)(pos_aux1_ - c0_2 + j)] = 2 + j;
  // stage 3: input = cat[x, aux1, aux2]       (lib/nets.py:75-77, 101-102)
  std::vector<int> p3((size_t)C3, -1);
  p3[(size_t)pos_x_] = 0; p3[(size_t)pos_x_ + 1] = 1;
  for (int j = 0; j < a1; ++j) p3[(size_t)(pos_aux1_ + j)] = 2 + j;
  for (int j = 0; j < a2; ++j) p3[(size_t)(pos_aux2_ + j)] = 2 + a1 + j;

  const int Hb = max_bin / 2;
  if (!build_basenet(nets_[0], "stg1_low_band_net.0", 2, p1, cp1, nout / 2, Hb, W, nin_lstm / 2, cfg_.nout_lstm))
    return false;
  if (!build_basenet(nets_[1], "stg1_high_band_net", 2, p1, cp1, nout / 4, Hb, W, nin_lstm / 2, cfg_.nout_lstm / 2))
    return false;
  if (!build_basenet(nets_[2], "stg2_low_band_net.0", a1 + 2, p2, cp2, nout, Hb, W, nin_lstm / 2, cfg_.nout_lstm))
    return false;
  if (!build_basenet(nets_[3], "stg2_high_band_net", a1 + 2, p2, cp2, nout / 2, Hb, W, nin_lstm / 2,
                     cfg_.nout_lstm / 2))
    return false;
  if (!build_basenet(nets_[4], "stg3_full_band_net", a1 + a2 + 2, p3, C3, nout, max_bin, W, nin_lstm, cfg_.nout_lstm))
    return false;
  if (!make_conv(bridge1_, "stg1_low_band_net.1", identity_perm(nout / 2, nout / 2), nout / 2, 1, 1, 1, 1, ACT_RELU))
    return false;
  if (!make_conv(bridge2_, "stg2_low_band_net.1", identity_perm(nout, nout), nout, 1, 1, 1, 1, ACT_RELU)) return false;
  const HostTensor *ow, *aw;
  if (!need("out.weight", {2, nout, 1, 1}, &ow)) return false;
  if (!need("aux_out.weight", {2, 3 * nout / 4, 1, 1}, &aw)) return false;   // dead in forward, but a strict key
  out_w_ = (float*)dalloc(sizeof(float) * 2 * nout);
  if (!out_w_) return false;
  cudaMemcpy(out_w_, ow->data.data(), sizeof(float) * 2 * nout, cudaMemcpyHostToDevice);
  // strict load: no unexpected keys (torch load_state_dict(strict=True), inference.py:131)
  {
    // every key outside the model's name space is unexpected
    for (auto& kv : sd_) {
      const std::string& k = kv.first;
      bool ok = k == "out.weight" || k == "aux_out.weight" || k.rfind("stg1_low_band_net.", 0) == 0 ||
                k.rfind("stg1_high_band_net.", 0) == 0 || k.rfind("stg2_low_band_net.", 0) == 0 ||
                k.rfind("stg2_high_band_net.", 0) == 0 || k.rfind("stg3_full_band_net.", 0) == 0;
      if (!ok) {
        err = "unexpected key in state_dict: " + k;
        return false;
      }
    }
  }
  if (!ck(cudaDeviceSynchronize(), "finalize")) return false;
  finalized_ = true;
  return true;
}

// ---------------------------------------------------------------------------------------------
void Engine::profile_enable(bool on) {
  for (auto& r : prof_) {
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  prof_.clear();
  profiling_ = on;
}

int Engine::prof_begin(const std::string& name, int kind, double flops, int N, int H, int W, cudaStream_t s) {
  if (!profiling_) return -1;
  ProfRec rec;
  cudaEventCreate(&rec.a);
  cudaEventCreate(&rec.b);
  rec.tc = kind; rec.flops = flops; rec.name = name;
  rec.N = N; rec.H = H; rec.W = W;
  cudaEventRecord(rec.a, s);
  prof_.push_back(rec);
  return (int)prof_.size() - 1;
}

void Engine::prof_end(int idx, cudaStream_t s) {
  if (idx >= 0) cudaEventRecord(prof_[(size_t)idx].b, s);
}

bool Engine::profile_read(double* out6) {
  for (int i = 0; i < 6; ++i) out6[i] = 0.0;
  for (auto& r : prof_) {
    if (r.tc > 1) continue;   // only the convolutions enter the roofline sums
    if (!ck(cudaEventSynchronize(r.b), "profile sync")) return false;
    float ms = 0.f;
    if (!ck(cudaEventElapsedTime(&ms, r.a, r.b), "profile elapsed")) return false;
    const int o = r.tc ? 0 : 3;
    out6[o] += ms;
    out6[o + 1] += r.flops;
    out6[o + 2] += 1.0;
  }
  return true;
}

bool Engine::profile_dump(std::string& text) {
  text.clear();
  char line[256];
  for (auto& r : prof_) {
    if (!ck(cudaEventSynchronize(r.b), "profile sync")) return false;
    float ms = 0.f;
    if (!ck(cudaEventElapsedTime(&ms, r.a, r.b), "profile elapsed")) return false;
    snprintf(line, sizeof(line), "%s %d %d %d %d %.6f %.6f\n", r.name.c_str(), r.N, r.H, r.W, r.tc, (double)ms,
             r.flops * 1e-9);
    text += line;
  }
  return true;
}

bool Engine::run_conv(ConvLayer& L, const ActView& in, const ActView& out, cudaStream_t s, const ActView* up_src,
                      const ActView* extra) {
  ++launches;
  const bool use_tc = L.tc && cfg_.conv_mode == 0 && tc_supported(L, in, out);
  if (!use_tc && cfg_.conv_mode == 0 && L.Cout >= 4 && !warned_simt_) {
    // loud, once per context: this geometry does not tile for the tcgen05 kernels (e.g. a cropsize whose feature-map
    // widths are not powers of two / multiples of 128) and runs on the fp32 CUDA-core kernel, an order of magnitude slower
    warned_simt_ = true;
    fprintf(stderr,
            "libvr_b200: WARNING: %s (N=%d, %dx%d -> %dx%d) does not tile for the tensor-core kernels and runs on the "
            "CUDA-core convolution; use a cropsize whose maps tile (e.g. 256) for full speed\n",
            L.name.c_str(), in.N, in.H, in.W, out.H, out.W);
  }
  // algorithmic FLOPs with the real (un-padded) channel counts: 2 * pixels * Cout * Cin * taps
  const int pi = prof_begin(up_src ? L.name + "+up" : L.name, use_tc ? 1 : 0,
                            2.0 * (double)out.N * out.H * out.W * L.Cout * L.Cin * L.k * L.k, out.N, out.H, out.W, s);
  bool ok = run_conv_inner(L, in, out, use_tc, s, up_src, extra);
  prof_end(pi, s);
  return ok;
}

bool Engine::run_conv_inner(ConvLayer& L, const ActView& in, const ActView& out, bool use_tc, cudaStream_t s,
                            const ActView* up_src, const ActView* extra) {
  if (use_tc) return ck(tc_launch(L, in, out, s, err, up_src, extra), L.name.c_str());
  if (up_src || extra) {
    err = "internal: fused upsample requested for a CUDA-core convolution";
    return false;
  }
  ConvParams p;
  p.in = in; p.out = out;
  p.w = L.w; p.bias = L.bias;
  p.CinPad = L.CinPad; p.Cout = L.Cout; p.CoutPad = L.CoutPad;
  p.KH = L.k; p.KW = L.k; p.stride = L.stride;
  p.dil_h = L.dil_h; p.dil_w = L.dil_w;
  p.pad_h = L.dil_h * (L.k / 2); p.pad_w = L.dil_w * (L.k / 2);
  p.act = L.act;
  p.in.C = L.CinPad;
  return ck(launch_conv_simt(p, s), L.name.c_str());
}

bool Engine::run_decoder(ConvLayer& L, const ActView& low, const Buffer& cat, int N, const ActView& out,
                         cudaStream_t s) {
  const ActView cat_all = cat.all(N);
  if (cfg_.conv_mode == 0 && L.tc && tc_supported(L, cat_all, out) && tc_can_fuse_upsample(L, cat_all, out, low))
    return run_conv(L, cat_all, out, s, &low);   // channels [0, low.C) of cat are produced inside the kernel
  if (cat.C < low.C + 1) {
    err = "internal: " + L.name + " was laid out for the fused upsample but the fused kernel is not available";
    return false;
  }
  ++launches;
  if (!timed("upsample2x", N, cat.H, cat.W, s, [&] { return ck(launch_upsample2x(low, cat.view(N, 0, cat.H, 0, low.C), s), "decoder upsample"); }))
    return false;
  return run_conv(L, cat_all, out, s);
}

bool Engine::run_basenet(BaseNetPlan& P, const ActView& in, const ActView& out, int N, cudaStream_t s,
                         cudaStream_t side) {
  const int n = P.n, H = P.H;
  // encoders (lib/nets.py:27-31); each skip tensor is written straight into its decoder's concat buffer
  ActView e1 = P.cat1.view(N, 0, H, P.e1_coff, n);
  if (!run_conv(P.enc1, in, e1, s)) return false;
  ActView e2 = P.cat2.view(N, 0, H / 2, 4 * n, 2 * n);
  if (!run_conv(P.enc_a[0], e1, P.t2.all(N), s) || !run_conv(P.enc_b[0], P.t2.all(N), e2, s)) return false;
  ActView e3 = P.cat3.view(N, 0, H / 4, 6 * n, 4 * n);
  if (!run_conv(P.enc_a[1], e2, P.t3.all(N), s) || !run_conv(P.enc_b[1], P.t3.all(N), e3, s)) return false;
  ActView e4 = P.cat4.view(N, 0, H / 8, 8 * n, 6 * n);
  if (!run_conv(P.enc_a[2], e3, P.t4.all(N), s) || !run_conv(P.enc_b[2], P.t4.all(N), e4, s)) return false;
  if (!run_conv(P.enc_a[3], e4, P.t5.all(N), s) || !run_conv(P.enc_b[3], P.t5.all(N), P.e5.all(N), s)) return false;
  // ASPP (lib/layers.py:92-105)
  const int c8 = 8 * n, h16 = H / 16;
  launches += 2;
  if (!timed("aspp.pool_freq_mean", N, h16, P.W / 16, s, [&] { return ck(launch_pool_freq_mean(P.e5.all(N), P.pool.all(N), s), "aspp pool"); }))
    return false;
  if (!run_conv(P.aspp1, P.pool.all(N), P.f1.all(N), s)) return false;
  if (!timed("aspp.broadcast_rows", N, h16, P.W / 16, s, [&] { return ck(launch_broadcast_rows(P.f1.all(N), P.acat.view(N, 0, h16, 0, c8), s), "aspp broadcast"); }))
    return false;
  if (!run_conv(P.aspp2, P.e5.all(N), P.acat.view(N, 0, h16, c8, c8), s)) return false;
  for (int i = 0; i < 3; ++i)
    if (!run_conv(P.aspp_d[i], P.e5.all(N), P.acat.view(N, 0, h16, (2 + i) * c8, c8), s)) return false;
  if (!run_conv(P.bott, P.acat.all(N), P.ao.all(N), s)) return false;
  // decoders (lib/nets.py:35-37, lib/layers.py:51-64)
  launches += 2;
  if (!timed("upsample2x", N, H / 8, P.W / 8, s, [&] { return ck(launch_upsample2x(P.ao.all(N), P.cat4.view(N, 0, H / 8, 0, 8 * n), s), "up4"); }))
    return false;
  if (!run_conv(P.dec[0], P.cat4.all(N), P.d4.all(N), s)) return false;
  if (!timed("upsample2x", N, H / 4, P.W / 4, s, [&] { return ck(launch_upsample2x(P.d4.all(N), P.cat3.view(N, 0, H / 4, 0, 6 * n), s), "up3"); }))
    return false;
  if (!run_conv(P.dec[1], P.cat3.all(N), P.d3.all(N), s)) return false;
  // The LSTM branch's 1x1 input convolution (2n -> 1, lib/layers.py:112,126) is one dot product per pixel of dec2's
  // output: the row kernel's epilogue accumulates it from the fp32 activations it is about to store.
  LstmPlan& Q = P.lstm;
  const ActView d2v = P.d2.view(N, 0, H / 2, 0, 2 * n);
  const bool dot_fused = cfg_.conv_mode == 0 && P.dec[2].tc && tc_supported(P.dec[2], P.cat2.all(N), d2v) &&
                         tc_rows_supported(P.dec[2], *P.dec[2].tc, P.cat2.all(N), d2v);
  if (dot_fused) {
    if (!ck(cudaMemsetAsync(Q.l0, 0, sizeof(float) * (size_t)N * Q.bins * Q.T, s), "lstm conv clear")) return false;
    P.dec[2].dot_w = Q.conv_w;
    P.dec[2].dot_out = Q.l0;
  }
  const bool dec2_ok = run_decoder(P.dec[2], P.d3.all(N), P.cat2, N, d2v, s);
  P.dec[2].dot_w = nullptr;
  P.dec[2].dot_out = nullptr;
  if (!dec2_ok) return false;
  // LSTM branch -> channel 2n of d2 (lib/nets.py:38, lib/layers.py:124-133).  Its 128-step recurrence keeps only
  // 2N CTAs busy, so when a side stream is free (stage 3) it runs there while the main stream upsamples the 2n
  // convolution channels of d2; only the LSTM channel's 16-channel group is upsampled after the join.
  const bool overlap = side != nullptr && !profiling_;
  cudaStream_t sl = overlap ? side : s;
  if (overlap) {
    if (!ck(cudaEventRecord(ev_lstm_fork_, s), "lstm fork") || !ck(cudaStreamWaitEvent(side, ev_lstm_fork_, 0), "lstm fork"))
      return false;
  }
  launches += dot_fused ? 3 : 4;
  if (!dot_fused &&
      !timed("lstm.inconv", N, H / 2, P.W / 2, sl, [&] { return ck(launch_lstm_inconv(d2v, Q.conv_w, Q.l0, sl), "lstm conv"); }))
    return false;
  if (!timed("lstm.input_projection", N, H / 2, P.W / 2, sl, [&] { return ck(launch_lstm_input_projection(Q.l0, Q.conv_bias, Q.wih, Q.bih, Q.xp, N, Q.T, Q.bins, 8 * Q.hid, sl), "lstm input projection"); }))
    return false;
  if (!timed("lstm.recurrence", N, H / 2, P.W / 2, sl, [&] { return ck(launch_lstm_recurrence(Q.xp, Q.whh, Q.hs, N, Q.T, Q.hid, sl), "lstm recurrence"); }))
    return false;
  // the branch output at half resolution: fp32 plane y[bin][n][t]
  if (!timed("lstm.dense", N, H / 2, P.W / 2, sl, [&] { return ck(launch_lstm_dense(Q.hs, Q.wd, Q.dscale, Q.dshift, N * Q.T, 2 * Q.hid, Q.bins, Q.y, sl), "lstm dense"); }))
    return false;
  ++launches;
  if (!P.skip_only &&   // staged layout: it becomes channel 2n of d2 and is up-sampled together with h
      !timed("lstm.to_channel", N, H / 2, P.W / 2, sl, [&] { return ck(launch_lstm_plane_to_channel(Q.y, N, Q.T, Q.bins, P.d2.all(N), 2 * n, sl), "lstm channel"); }))
    return false;
  if (P.skip_only) {
    // fused layout: up(lstm) -> its 16-channel group of cat1 / lstm_up (small kernel on the LSTM's stream), then the row
    // kernel reads [e1 | up(lstm)] by TMA and produces up(h) itself from d2
    const ActView lstm_full = P.lstm_own ? P.lstm_up.all(N) : P.cat1.view(N, 0, H, P.lstm_coff, 16);
    if (!timed("lstm.upsample2x", N, H, P.W, sl, [&] { return ck(launch_upsample2x_c1(Q.y, Q.bins, Q.T, Q.T, (int64_t)N * Q.T, lstm_full, sl), "lstm upsample"); }))
      return false;
    if (overlap) {
      if (!ck(cudaEventRecord(ev_lstm_join_, side), "lstm join") || !ck(cudaStreamWaitEvent(s, ev_lstm_join_, 0), "lstm join"))
        return false;
    }
    const ActView h = P.d2.all(N);
    if (!tc_can_fuse_upsample(P.dec[3], P.cat1.all(N), out, h)) {
      err = "internal: " + P.prefix + ".dec1 was laid out for the fused upsample but the fused kernel is not available";
      return false;
    }
    return run_conv(P.dec[3], P.cat1.all(N), out, s, &h, P.lstm_own ? &lstm_full : nullptr);
  }
  // staged layout: dec1 on cat[up(h, lstm), e1] (lib/nets.py:39)
  const int upc = P.e1_off;   // channels of d2 that are upsampled: 2n conv channels + the LSTM channel group
  if (overlap) {
    if (!ck(cudaEventRecord(ev_lstm_join_, side), "lstm join")) return false;
    if (cfg_.conv_mode == 0 && tc_can_fuse_upsample(P.dec[3], P.cat1.all(N), out, P.d2.all(N))) {
      // fused: the convolution reads d2 (incl. the LSTM channel) itself, so it simply waits for the side stream
      if (!ck(cudaStreamWaitEvent(s, ev_lstm_join_, 0), "lstm join")) return false;
      return run_decoder(P.dec[3], P.d2.all(N), P.cat1, N, out, s);
    }
    ++launches;
    if (!ck(launch_upsample2x(P.d2.view(N, 0, H / 2, 0, 2 * n), P.cat1.view(N, 0, H, 0, 2 * n), s), "up1")) return false;
    if (!ck(cudaStreamWaitEvent(s, ev_lstm_join_, 0), "lstm join")) return false;
    if (!ck(launch_upsample2x(P.d2.view(N, 0, H / 2, 2 * n, upc - 2 * n), P.cat1.view(N, 0, H, 2 * n, upc - 2 * n), s),
            "up1 lstm"))
      return false;
    return run_conv(P.dec[3], P.cat1.all(N), out, s);
  }
  return run_decoder(P.dec[3], P.d2.all(N), P.cat1, N, out, s);
}

bool Engine::forward(int N, cudaStream_t s) {
  const int max_bin = cfg_.n_fft / 2, Hb = max_bin / 2;
  const int nout = cfg_.nout, a1 = nout / 4, a2 = nout / 2;
  const int c0_1 = pos_x_ / 16 * 16, c0_2 = pos_aux1_ / 16 * 16;
  last_n_ = N;
  // Stages 1 and 2 (lib/nets.py:91-99): the low-band chain (stg1_low -> bridge -> stg2_low -> bridge) and the
  // high-band chain (stg1_high -> stg2_high) only meet at stage 3, so they run on two streams.
  const bool two = s_hi_ != nullptr && !profiling_;
  cudaStream_t sh = two ? s_hi_ : s;
  if (two) {
    if (!ck(cudaEventRecord(ev_fork_, s), "fork") || !ck(cudaStreamWaitEvent(s_hi_, ev_fork_, 0), "fork wait"))
      return false;
  }
  if (!run_basenet(nets_[1], in3_.view(N, Hb, Hb, c0_1, nets_[1].enc1.CinPad), in3_.view(N, Hb, Hb, pos_aux1_, a1), N,
                   sh))
    return false;
  if (!run_basenet(nets_[3], in3_.view(N, Hb, Hb, c0_2, nets_[3].enc1.CinPad), in3_.view(N, Hb, Hb, pos_aux2_, a2), N,
                   sh))
    return false;
  if (!run_basenet(nets_[0], in3_.view(N, 0, Hb, c0_1, nets_[0].enc1.CinPad), o1_.all(N), N, s)) return false;
  if (!run_conv(bridge1_, o1_.all(N), in3_.view(N, 0, Hb, pos_aux1_, a1), s)) return false;
  if (!run_basenet(nets_[2], in3_.view(N, 0, Hb, c0_2, nets_[2].enc1.CinPad), o2_.all(N), N, s)) return false;
  if (!run_conv(bridge2_, o2_.all(N), in3_.view(N, 0, Hb, pos_aux2_, a2), s)) return false;
  if (two) {
    if (!ck(cudaEventRecord(ev_join_, s_hi_), "join") || !ck(cudaStreamWaitEvent(s, ev_join_, 0), "join wait"))
      return false;
  }
  // stage 3 (lib/nets.py:101-102)
  return run_basenet(nets_[4], in3_.all(N), f3_.all(N), N, s, two ? s_hi_ : nullptr);
}

// ---------------------------------------------------------------------------------------------
bool Engine::predict_mask(const float* mag, int N, float* mask_out, int offset, cudaStream_t s) {
  if (!finalized_) {
    err = "weights not finalized";
    return false;
  }
  cudaSetDevice(cfg_.device);
  const int max_bin = cfg_.n_fft / 2, nb = bins(), W = cfg_.cropsize, r = W - 2 * offset;
  for (int i = 0; i < N; i += cfg_.max_batch) {
    const int nb_now = N - i < cfg_.max_batch ? N - i : cfg_.max_batch;
    ++launches;
    if (!ck(launch_pack_mag_from_float(mag + (int64_t)i * 2 * nb * W, nb, max_bin,
                                       in3_.view(nb_now, 0, max_bin, pos_x_, 2), s),
            "pack"))
      return false;
    if (!forward(nb_now, s)) return false;
    MaskOutParams p;
    p.f3 = f3_.all(nb_now);
    p.w = out_w_;
    p.out = mask_out + (int64_t)i * 2 * nb * r;
    p.stride_n = (int64_t)2 * nb * r; p.stride_c = (int64_t)nb * r; p.stride_bin = r;
    p.offset = offset; p.t_base0 = 0; p.t_limit = r; p.roi_t = 0; p.accumulate = 0;
    ++launches;
    if (!timed("mask_out", nb_now, max_bin, W, s, [&] { return ck(launch_mask_out(p, s), "mask_out"); })) return false;
  }
  return true;
}

bool Engine::separate_windows(const float2* spec, int64_t T, const float* norm, int pad_l, int first, int count,
                              float* mask, int64_t mask_T, int64_t frame_shift, int accumulate, cudaStream_t s,
                              bool final_pass) {
  if (!finalized_) {
    err = "weights not finalized";
    return false;
  }
  cudaSetDevice(cfg_.device);
  const int max_bin = cfg_.n_fft / 2, nb = bins(), W = cfg_.cropsize, r = roi();
  for (int i = 0; i < count; i += cfg_.max_batch) {
    const int n_now = count - i < cfg_.max_batch ? count - i : cfg_.max_batch;
    const int g0 = first + i;
    ++launches;
    if (!timed("pack_mag_from_spec", n_now, max_bin, W, s, [&] {
          return ck(launch_pack_mag_from_spec(spec, nb, T, max_bin, W, r, pad_l, g0, norm, in3_.view(n_now, 0, max_bin, pos_x_, 2), s), "pack");
        }))
      return false;
    if (!forward(n_now, s)) return false;
    MaskOutParams p;
    p.f3 = f3_.all(n_now);
    p.w = out_w_;
    p.out = mask;
    p.stride_n = r; p.stride_c = (int64_t)nb * mask_T; p.stride_bin = mask_T;
    p.offset = cfg_.offset;
    p.t_base0 = (int64_t)g0 * r - frame_shift;
    p.t_limit = mask_T; p.roi_t = r; p.accumulate = accumulate;
    ++launches;
    if (!timed("mask_out", n_now, max_bin, W, s, [&] { return ck(launch_mask_out(p, s), "mask_out"); })) return false;
    if (final_pass && on_frames_final_) {
      int64_t f = p.t_base0 + (int64_t)n_now * r;
      if (f > mask_T) f = mask_T;
      if (f > 0 && !on_frames_final_(f)) return false;
    }
  }
  return true;
}

bool Engine::normaliser(const float2* spec, int64_t T, int mode, float* out, cudaStream_t s) {
  cudaSetDevice(cfg_.device);
  ++launches;
  const int64_t n = (int64_t)2 * bins() * T;
  if (mode == 0) return timed("normaliser.absmax", 1, bins(), (int)T, s, [&] { return ck(launch_absmax(spec, n, out, s), "absmax"); });
  return timed("normaliser.lexmax", 1, bins(), (int)T, s, [&] { return ck(launch_lexmax_abs(spec, n, ws_lex_, out, s), "lexmax"); });
}

// mask [2][bins][T]; the full window range of one track on this device (inference.py:70-77 / 83-98)
bool Engine::separate(const float2* spec, int64_t T, int tta, float* mask, cudaStream_t s) {
  const int r = roi();
  const int pad_l = cfg_.offset;
  // make_padding (lib/dataset.py:198-205): right = roi - (T % roi) + left
  const int64_t pad_r = r - (T % r) + pad_l;
  const int64_t Wpad = pad_l + T + pad_r;
  const int patches = (int)((Wpad - 2 * cfg_.offset) / r);
  if (!normaliser(spec, T, tta ? 1 : 0, ws_norm_, s)) return false;
  if (!separate_windows(spec, T, ws_norm_, pad_l, 0, patches, mask, T, 0, 0, s, !tta)) return false;
  if (tta) {
    const int64_t Wpad2 = Wpad + r;   // pad_l += roi/2, pad_r += roi/2 (inference.py:91-92)
    const int patches2 = (int)((Wpad2 - 2 * cfg_.offset) / r);
    if (!separate_windows(spec, T, ws_norm_, pad_l + r / 2, 0, patches2, mask, T, r / 2, 1, s, true)) return false;
  }
  return true;
}

bool Engine::apply_mask(const float2* spec, const float* mask, int64_t T, float2* y, float2* v, cudaStream_t s) {
  cudaSetDevice(cfg_.device);
  ++launches;
  return ck(launch_apply_mask(spec, mask, (int64_t)2 * bins() * T, y, v, s), "apply_mask");
}

bool Engine::stft(const float* wave, int64_t L, float2* spec, int64_t T, float* absmax, cudaStream_t s) {
  if (!stft_range(wave, L, spec, T, 0, T, s)) return false;
  if (absmax) return normaliser(spec, T, 0, absmax, s);
  return true;
}

// frames [t0, t1) of the track only: what a rank of the window-sharded path needs (lib/distributed.py)
bool Engine::stft_range(const float* wave, int64_t L, float2* spec, int64_t T, int64_t t0, int64_t t1, cudaStream_t s) {
  cudaSetDevice(cfg_.device);
  if (T != 1 + L / cfg_.hop) {
    err = "stft: T must equal 1 + L // hop_length";
    return false;
  }
  if (t0 < 0 || t1 > T || t0 > t1) {
    err = "stft: frame range outside [0, T]";
    return false;
  }
  ++launches;
  return timed("stft", 1, bins(), (int)(t1 - t0), s, [&] { return ck(launch_stft(wave, L, cfg_.n_fft, cfg_.hop, spec, T, t0, t1, twiddle_, window_, s), "stft"); });
}

bool Engine::normaliser_range(const float2* spec, int64_t T, int64_t t0, int64_t t1, float* out, cudaStream_t s) {
  cudaSetDevice(cfg_.device);
  if (t0 < 0 || t1 > T || t0 > t1) {
    err = "normaliser: frame range outside [0, T]";
    return false;
  }
  ++launches;
  return ck(launch_absmax_range(spec, 2 * bins(), T, t0, t1, out, s), "absmax range");
}

bool Engine::ensure_ws(int64_t T) {
  const int64_t nspec = (int64_t)2 * bins() * T;
  if (nspec > ws_spec_cap_) {
    if (ws_spec_) cudaFree(ws_spec_);
    ws_spec_ = nullptr;
    if (!ck(cudaMalloc(&ws_spec_, sizeof(float2) * nspec), "workspace spec")) return false;
    ws_spec_cap_ = nspec;
  }
  if (nspec > ws_mask_cap_) {
    if (ws_mask_) cudaFree(ws_mask_);
    ws_mask_ = nullptr;
    if (!ck(cudaMalloc(&ws_mask_, sizeof(float) * nspec), "workspace mask")) return false;
    ws_mask_cap_ = nspec;
  }
  const int64_t nfr = (int64_t)4 * T * cfg_.n_fft;
  if (nfr > ws_frames_cap_) {
    if (ws_frames_) cudaFree(ws_frames_);
    ws_frames_ = nullptr;
    if (!ck(cudaMalloc(&ws_frames_, sizeof(float) * nfr), "workspace frames")) return false;
    ws_frames_cap_ = nfr;
  }
  return true;
}

bool Engine::istft(const float2* spec, const float* mask, int64_t T, float* wave_a, float* wave_b, cudaStream_t s) {
  return istft_range(spec, mask, T, 0, T - 1, wave_a, wave_b, s);
}

// Output hops [k0, k1) (samples [hop*k0, hop*k1)) of wave [2][hop*(T-1)]; reads frames of spec / mask that overlap
// them (k0 - n_fft/hop/2 + 1 .. k1 + n_fft/hop/2 - 1 clipped to the track; k0..k1 for hop = n_fft/2).
// wave_a / wave_b may point into another GPU's memory (peer-mapped).
bool Engine::istft_range(const float2* spec, const float* mask, int64_t T, int64_t k0, int64_t k1, float* wave_a,
                         float* wave_b, cudaStream_t s) {
  cudaSetDevice(cfg_.device);
  if (k0 < 0 || k1 > T - 1 || k0 > k1) {
    err = "istft: hop range outside [0, T-1]";
    return false;
  }
  if (k1 == k0) return true;
  const int NF = cfg_.n_fft, hop = cfg_.hop;
  // first / last frame touching samples [hop*k0, hop*k1): u = s + NF/2, frames ceil((u-NF+1)/hop) .. floor(u/hop)
  int64_t f0 = ((int64_t)hop * k0 + NF / 2 - NF + hop) / hop;
  if ((int64_t)hop * k0 + NF / 2 - NF + 1 <= 0) f0 = 0;
  int64_t f1 = ((int64_t)hop * k1 - 1 + NF / 2) / hop;
  if (f1 > T - 1) f1 = T - 1;
  const int64_t nfr = f1 - f0 + 1;
  const int64_t need = (int64_t)4 * nfr * NF;
  if (need > ws_frames_cap_) {
    if (ws_frames_) cudaFree(ws_frames_);
    ws_frames_ = nullptr;
    if (!ck(cudaMalloc(&ws_frames_, sizeof(float) * need), "workspace frames")) return false;
    ws_frames_cap_ = need;
  }
  float* fa = ws_frames_;
  float* fb = mask ? ws_frames_ + (int64_t)2 * nfr * NF : nullptr;
  launches += 2;
  if (!timed("istft.frames", 1, bins(), (int)nfr, s, [&] { return ck(launch_istft_frames(spec, mask, NF, T, f0, nfr, fa, fb, twiddle_, window_, s), "istft frames"); }))
    return false;
  return timed("istft.overlap_add", 1, bins(), (int)nfr, s, [&] {
    return ck(launch_istft_ola(fa, fb, NF, hop, T, f0, nfr, (int64_t)hop * k0, (int64_t)hop * k1, wave_a, mask ? wave_b : nullptr, window_, s), "istft ola");
  });
}

// wave (2, L) in HBM -> instruments / vocals waves (2, hop*(T-1)) in HBM: the whole inference.py:147-176 path.
bool Engine::separate_wave(const float* wave, int64_t L, int tta, float* inst, float* voc, cudaStream_t s) {
  cudaSetDevice(cfg_.device);
  const int64_t T = 1 + L / cfg_.hop;
  if (!ensure_ws(T)) return false;
  if (!stft(wave, L, ws_spec_, T, nullptr, s)) return false;
  if (!separate(ws_spec_, T, tta, ws_mask_, s)) return false;
  return istft(ws_spec_, ws_mask_, T, inst, voc, s);
}

// Host-buffer entry (the end-to-end call): H2D of the wave, the whole path, D2H of both stems.
bool Engine::separate_wave_host(const float* wave, int64_t L, int tta, float* inst, float* voc, cudaStream_t s) {
  cudaSetDevice(cfg_.device);
  const int64_t T = 1 + L / cfg_.hop;
  const int64_t Lo = (int64_t)cfg_.hop * (T - 1);
  const int64_t need_f = 2 * L + 4 * Lo;
  if (need_f > ws_wave_cap_) {
    if (ws_wave_) cudaFree(ws_wave_);
    ws_wave_ = nullptr;
    if (!ck(cudaMalloc(&ws_wave_, sizeof(float) * need_f), "workspace wave")) return false;
    ws_wave_cap_ = need_f;
  }
  float* d_in = ws_wave_;
  float* d_inst = ws_wave_ + 2 * L;
  float* d_voc = d_inst + 2 * Lo;
  if (!ck(cudaMemcpyAsync(d_in, wave, sizeof(float) * 2 * L, cudaMemcpyHostToDevice, s), "H2D wave")) return false;
  // The stems leave the device span by span: as soon as a window batch of the last pass has written its mask frames,
  // the masked inverse STFT of the hops they complete runs on `s` and their device-to-host copy on the copy stream,
  // overlapped with the next batch of the net (the copies of a 4-minute track are 169 MB).
  if (!ensure_ws(T)) return false;
  if (!stft(d_in, L, ws_spec_, T, nullptr, s)) return false;
  int64_t k_done = 0;
  bool ok = true;
  auto flush = [&](int64_t f) -> bool {
    // output hop k needs mask frames k and k+1
    int64_t k1 = f >= T ? T - 1 : f - 1;
    if (k1 <= k_done) return true;
    if (!istft_range(ws_spec_, ws_mask_, T, k_done, k1, d_inst, d_voc, s)) return false;
    if (!ck(cudaEventRecord(ev_span_, s), "span event") || !ck(cudaStreamWaitEvent(s_copy_, ev_span_, 0), "span wait"))
      return false;
    const size_t off = (size_t)cfg_.hop * (size_t)k_done, cnt = (size_t)cfg_.hop * (size_t)(k1 - k_done);
    for (int c = 0; c < 2; ++c) {
      if (!ck(cudaMemcpyAsync(inst + (size_t)c * Lo + off, d_inst + (size_t)c * Lo + off, sizeof(float) * cnt,
                              cudaMemcpyDeviceToHost, s_copy_), "D2H inst") ||
          !ck(cudaMemcpyAsync(voc + (size_t)c * Lo + off, d_voc + (size_t)c * Lo + off, sizeof(float) * cnt,
                              cudaMemcpyDeviceToHost, s_copy_), "D2H voc"))
        return false;
    }
    k_done = k1;
    return true;
  };
  on_frames_final_ = flush;
  ok = separate(ws_spec_, T, tta, ws_mask_, s);
  on_frames_final_ = nullptr;
  if (ok) ok = flush(T);
  if (!ok) {
    cudaStreamSynchronize(s);
    cudaStreamSynchronize(s_copy_);
    return false;
  }
  return ck(cudaStreamSynchronize(s), "separate_wave_host sync") && ck(cudaStreamSynchronize(s_copy_), "separate_wave_host copy sync");
}

// ---------------------------------------------------------------------------------------------
// Several tracks per call.  Windows are independent inside the net (eval-mode BatchNorm, per-sample ASPP pool and
// LSTM), so windows of different tracks share a forward batch without changing any arithmetic; only the gather into
// the input buffer, the mask epilogue and the normalisers read per-track tables.
bool Engine::ensure_norms(int n) {
  if (n <= ws_norms_cap_) return true;
  if (ws_norms_) cudaFree(ws_norms_);
  if (ws_lexs_) cudaFree(ws_lexs_);
  ws_norms_ = nullptr;
  ws_lexs_ = nullptr;
  ws_norms_cap_ = 0;
  if (!ck(cudaMalloc(&ws_norms_, sizeof(float) * n), "workspace normalisers") ||
      !ck(cudaMalloc(&ws_lexs_, sizeof(unsigned long long) * n), "workspace lexmax"))
    return false;
  ws_norms_cap_ = n;
  return true;
}

bool Engine::upload_tables(const Tables& t, cudaStream_t s, const unsigned char** dev) {
  const size_t nb = t.bytes.size() ? t.bytes.size() : 16;
  // the previous call's copy out of the pinned buffer must have run before the buffer is rewritten
  if (!ck(cudaEventSynchronize(ev_tab_copied_), "tables: previous copy")) return false;
  if (nb > tab_host_cap_) {
    if (tab_host_) cudaFreeHost(tab_host_);
    tab_host_ = nullptr;
    tab_host_cap_ = 0;
    if (!ck(cudaMallocHost(&tab_host_, nb), "tables: pinned buffer")) return false;
    tab_host_cap_ = nb;
  }
  if (nb > tab_dev_cap_) {
    if (!ck(cudaEventSynchronize(ev_tab_used_), "tables: previous call")) return false;
    if (tab_dev_) cudaFree(tab_dev_);
    tab_dev_ = nullptr;
    tab_dev_cap_ = 0;
    if (!ck(cudaMalloc(&tab_dev_, nb), "tables: device buffer")) return false;
    tab_dev_cap_ = nb;
  }
  if (!t.bytes.empty()) memcpy(tab_host_, t.bytes.data(), t.bytes.size());
  // the previous call's kernels read the device table: the stream waits for them, the host does not
  if (!ck(cudaStreamWaitEvent(s, ev_tab_used_, 0), "tables: wait") ||
      !ck(cudaMemcpyAsync(tab_dev_, tab_host_, nb, cudaMemcpyHostToDevice, s), "tables: copy") ||
      !ck(cudaEventRecord(ev_tab_copied_, s), "tables: record"))
    return false;
  *dev = tab_dev_;
  return true;
}

// Pass 1 of every track follows make_padding (lib/dataset.py:198-205) as separate() does; with tta, pass 2 of every
// track uses pad_l + roi/2 and averages into the mask (inference.py:89-98).  All pass-1 windows of all tracks come
// first, then all pass-2 windows, cut into batches of max_batch.
//
// TTA ordering: a pass-2 window averages ((old + new) * 0.5) into mask frames that pass-1 windows of the SAME track
// wrote.  Within one mask-epilogue launch there is no order between windows, so a batch must never hold a pass-2
// window of a track together with a pass-1 window of that track: at the pass boundary such a batch is closed early.
// (Windows of one pass write disjoint frames, and batches run in stream order.)
void Engine::schedule_windows(const float2* const* specs, const int64_t* T, int n, int tta, float* const* masks,
                              Schedule& sch) const {
  const int r = roi(), off = cfg_.offset, B = cfg_.max_batch;
  sch.wins.clear();
  sch.chunk_end.clear();
  for (int pass = 0; pass < (tta ? 2 : 1); ++pass) {
    for (int i = 0; i < n; ++i) {
      const int64_t pad_r = r - (T[i] % r) + off;
      const int64_t Wpad = off + T[i] + pad_r + (pass ? r : 0);   // pass 2: pad_l += roi/2, pad_r += roi/2
      const int patches = (int)((Wpad - 2 * off) / r);
      for (int g = 0; g < patches; ++g) {
        WinDesc d;
        d.spec = specs[i];
        d.mask = masks[i];
        d.T = T[i];
        d.t_base = (int64_t)g * r - (pass ? r / 2 : 0);
        d.pad_l = off + (pass ? r / 2 : 0);
        d.window = g;
        d.norm = i;
        d.accumulate = pass;
        sch.wins.push_back(d);
      }
    }
  }
  std::vector<char> pass1_in_batch((size_t)n, 0);
  int start = 0;
  for (int k = 0; k < (int)sch.wins.size(); ++k) {
    const WinDesc& d = sch.wins[(size_t)k];
    if (k - start == B || (d.accumulate && pass1_in_batch[(size_t)d.norm])) {
      sch.chunk_end.push_back(k);
      for (int j = start; j < k; ++j) pass1_in_batch[(size_t)sch.wins[(size_t)j].norm] = 0;
      start = k;
    }
    if (!d.accumulate) pass1_in_batch[(size_t)d.norm] = 1;
  }
  if (start < (int)sch.wins.size()) sch.chunk_end.push_back((int)sch.wins.size());
}

// one table-driven pack, the forward and one table-driven mask epilogue per batch; norms in ws_norms_
bool Engine::run_schedule(const Schedule& sch, const WinDesc* d_wins, cudaStream_t s) {
  const int max_bin = cfg_.n_fft / 2, nb = bins(), W = cfg_.cropsize, r = roi();
  int start = 0;
  for (int end : sch.chunk_end) {
    const int n_now = end - start;
    const WinDesc* d = d_wins + start;
    ++launches;
    if (!timed("pack_mag_many", n_now, max_bin, W, s, [&] {
          return ck(launch_pack_mag_many(d, nb, max_bin, W, r, ws_norms_, in3_.view(n_now, 0, max_bin, pos_x_, 2), s), "pack many");
        }))
      return false;
    if (!forward(n_now, s)) return false;
    ++launches;
    if (!timed("mask_out_many", n_now, max_bin, W, s, [&] { return ck(launch_mask_out_many(f3_.all(n_now), out_w_, cfg_.offset, d, s), "mask_out many"); }))
      return false;
    start = end;
  }
  return true;
}

bool Engine::normalisers_many(const NormTrack* d_tracks, int n, int64_t max_n, int mode, cudaStream_t s) {
  ++launches;
  return timed(mode == 0 ? "normaliser.absmax_many" : "normaliser.lexmax_many", n, bins(), 0, s, [&] {
    return ck(launch_normaliser_many(d_tracks, n, max_n, mode, ws_lexs_, ws_norms_, s), "normalisers");
  });
}

bool Engine::separate_many(const float2* const* specs, const int64_t* T, int n, int tta, float* const* masks,
                           cudaStream_t s) {
  if (!finalized_) {
    err = "weights not finalized";
    return false;
  }
  cudaSetDevice(cfg_.device);
  if (!ensure_norms(n)) return false;
  std::vector<NormTrack> nt((size_t)n);
  int64_t max_n = 0;
  for (int i = 0; i < n; ++i) {
    nt[(size_t)i].spec = specs[i];
    nt[(size_t)i].n = (int64_t)2 * bins() * T[i];
    if (nt[(size_t)i].n > max_n) max_n = nt[(size_t)i].n;
  }
  Schedule sch;
  schedule_windows(specs, T, n, tta, masks, sch);
  Tables tab;
  const size_t o_norm = tab.put(nt), o_wins = tab.put(sch.wins);
  const unsigned char* d = nullptr;
  if (!upload_tables(tab, s, &d)) return false;
  if (!normalisers_many((const NormTrack*)(d + o_norm), n, max_n, tta ? 1 : 0, s)) return false;
  if (!run_schedule(sch, (const WinDesc*)(d + o_wins), s)) return false;
  return ck(cudaEventRecord(ev_tab_used_, s), "tables: record use");
}

// waves[i] (2, L[i]) -> inst[i], voc[i] (2, hop*(T_i-1)): ragged STFT into the concatenated spectrogram workspace,
// per-track normalisers, the packed windows, ragged masked inverse STFT.  One table upload for the whole call.
bool Engine::separate_waves(const float* const* waves, const int64_t* L, int n, int tta, float* const* inst,
                            float* const* voc, cudaStream_t s) {
  if (!finalized_) {
    err = "weights not finalized";
    return false;
  }
  cudaSetDevice(cfg_.device);
  const int NF = cfg_.n_fft, hop = cfg_.hop, nb = bins();
  std::vector<int64_t> T((size_t)n);
  int64_t sumT = 0;
  for (int i = 0; i < n; ++i) {
    T[(size_t)i] = 1 + L[i] / hop;
    sumT += T[(size_t)i];
  }
  if (!ensure_ws(sumT) || !ensure_norms(n)) return false;
  std::vector<FftTrack> ft((size_t)n);
  std::vector<NormTrack> nt((size_t)n);
  std::vector<const float2*> specs((size_t)n);
  std::vector<float*> masks((size_t)n);
  int64_t frames = 0, ctas = 0, samples = 0, max_n = 0;
  for (int i = 0; i < n; ++i) {
    const int64_t Ti = T[(size_t)i];
    FftTrack& f = ft[(size_t)i];
    f.wave = waves[i];
    f.spec = ws_spec_ + (int64_t)2 * nb * frames;
    f.mask = ws_mask_ + (int64_t)2 * nb * frames;
    f.wave_a = inst[i];
    f.wave_b = voc[i];
    f.L = L[i];
    f.T = Ti;
    f.frame_off = frames;
    f.cta0 = ctas;
    f.s0 = samples;
    frames += Ti;
    ctas += fft_ctas_per_track(NF, Ti);
    samples += (int64_t)2 * hop * (Ti - 1);
    specs[(size_t)i] = f.spec;
    masks[(size_t)i] = ws_mask_ + (int64_t)2 * nb * f.frame_off;
    nt[(size_t)i].spec = f.spec;
    nt[(size_t)i].n = (int64_t)2 * nb * Ti;
    if (nt[(size_t)i].n > max_n) max_n = nt[(size_t)i].n;
  }
  Schedule sch;
  schedule_windows(specs.data(), T.data(), n, tta, masks.data(), sch);
  Tables tab;
  const size_t o_fft = tab.put(ft), o_norm = tab.put(nt), o_wins = tab.put(sch.wins);
  const unsigned char* d = nullptr;
  if (!upload_tables(tab, s, &d)) return false;
  const FftTrack* d_ft = (const FftTrack*)(d + o_fft);
  ++launches;
  if (!timed("stft_many", n, nb, (int)frames, s, [&] { return ck(launch_stft_many(d_ft, n, ctas, NF, hop, twiddle_, window_, s), "stft many"); }))
    return false;
  if (!normalisers_many((const NormTrack*)(d + o_norm), n, max_n, tta ? 1 : 0, s)) return false;
  if (!run_schedule(sch, (const WinDesc*)(d + o_wins), s)) return false;
  float* fa = ws_frames_;
  float* fb = ws_frames_ + (int64_t)2 * frames * NF;
  launches += 2;
  if (!timed("istft.frames_many", n, nb, (int)frames, s, [&] { return ck(launch_istft_frames_many(d_ft, n, ctas, NF, fa, fb, twiddle_, window_, s), "istft frames many"); }))
    return false;
  if (!timed("istft.overlap_add_many", n, nb, (int)frames, s, [&] { return ck(launch_istft_ola_many(d_ft, n, samples, NF, hop, fa, fb, window_, s), "istft ola many"); }))
    return false;
  return ck(cudaEventRecord(ev_tab_used_, s), "tables: record use");
}

// ---------------------------------------------------------------------------------------------
bool Engine::debug_conv(const float* x_nchw, int N, int Cin, int H, int W, const float* w, const float* bias, int Cout,
                        int k, int stride, int dil_h, int dil_w, int act, int use_tc, float* y_nchw, cudaStream_t s) {
  cudaSetDevice(cfg_.device);
  const int cin_pad = round_up(Cin, 16);
  const int Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1;
  std::vector<void*> tmp;
  std::swap(tmp, allocs_);
  Buffer bin = make_buffer(N, H, W, cin_pad);
  Buffer bout = make_buffer(N, Ho, Wo, round_up(Cout, 8));
  ConvLayer L;
  L.name = "debug_conv";
  L.rows_wide = g_tc_debug[2] == 1;   // vr_debug_set(2, 1): exercise the 64-wide row tile on a plain convolution
  L.Cin = Cin; L.CinPad = cin_pad; L.Cout = Cout; L.CoutPad = round_up(Cout, 8);
  L.k = k; L.stride = stride; L.dil_h = dil_h; L.dil_w = dil_w; L.act = act;
  const int taps = k * k;
  std::vector<float> hw((size_t)Cout * Cin * taps), hb((size_t)Cout);
  cudaMemcpyAsync(hw.data(), w, hw.size() * sizeof(float), cudaMemcpyDeviceToHost, s);
  cudaMemcpyAsync(hb.data(), bias, hb.size() * sizeof(float), cudaMemcpyDeviceToHost, s);
  cudaStreamSynchronize(s);
  L.w_host.assign((size_t)taps * L.CinPad * L.CoutPad, 0.f);
  L.bias_host.assign((size_t)L.CoutPad, 0.f);
  for (int co = 0; co < Cout; ++co) {
    L.bias_host[(size_t)co] = hb[(size_t)co];
    for (int ci = 0; ci < Cin; ++ci)
      for (int t = 0; t < taps; ++t)
        L.w_host[((size_t)t * L.CinPad + ci) * L.CoutPad + co] = hw[((size_t)co * Cin + ci) * taps + t];
  }
  L.w = (float*)dalloc(L.w_host.size() * sizeof(float));
  L.bias = (float*)dalloc(L.bias_host.size() * sizeof(float));
  bool ok = bin.hi && bout.hi && L.w && L.bias;
  if (ok) {
    cudaMemcpy(L.w, L.w_host.data(), L.w_host.size() * sizeof(float), cudaMemcpyHostToDevice);
    cudaMemcpy(L.bias, L.bias_host.data(), L.bias_host.size() * sizeof(float), cudaMemcpyHostToDevice);
    ok = ck(launch_nchw_to_act(x_nchw, Cin, bin.all(N), s), "nchw_to_act");
  }
  const int saved_mode = cfg_.conv_mode;
  if (ok && use_tc) {
    ok = tc_prepare(L, err, allocs_);
    if (ok && !(L.tc && tc_supported(L, bin.all(N), bout.view(N, 0, Ho, 0, Cout)))) {
      err = "debug_conv: geometry not supported by the tcgen05 kernel";
      ok = false;
    }
    cfg_.conv_mode = 0;
  } else {
    cfg_.conv_mode = 1;
  }
  if (ok) ok = run_conv(L, bin.all(N), bout.view(N, 0, Ho, 0, Cout), s);
  cfg_.conv_mode = saved_mode;
  if (ok) ok = ck(launch_act_to_nchw(bout.view(N, 0, Ho, 0, Cout), Cout, y_nchw, s), "act_to_nchw");
  if (ok) ok = ck(cudaStreamSynchronize(s), "debug_conv sync");
  L.tc.reset();
  for (void* p : allocs_) cudaFree(p);
  allocs_.clear();
  std::swap(tmp, allocs_);
  return ok;
}

// Test hook for the decoder path: y = act(conv3x3(cat[up2x(low), skip]) + bias), fused (upsample inside the row
// kernel) or staged (upsample kernel, then convolution).
bool Engine::debug_decoder(const float* low_nchw, int N, int Cl, int h, int w, const float* skip_nchw, int Cs,
                           const float* wgt, const float* bias, int Cout, int act, int fused, float* y_nchw,
                           cudaStream_t s) {
  cudaSetDevice(cfg_.device);
  const int H = 2 * h, W = 2 * w, Cin = Cl + Cs;
  const int cl_pad = round_up(Cl, 32), cin_pad = round_up(cl_pad + Cs, 16);
  std::vector<void*> tmp;
  std::swap(tmp, allocs_);
  Buffer blow = make_buffer(N, h, w, cl_pad);
  Buffer bcat = make_buffer(N, H, W, cin_pad);
  Buffer bout = make_buffer(N, H, W, round_up(Cout, 16));
  ConvLayer L;
  L.name = "debug_decoder";
  L.rows_wide = true;
  L.Cin = Cin; L.CinPad = cin_pad; L.Cout = Cout; L.CoutPad = round_up(Cout, 8);
  L.k = 3; L.stride = 1; L.dil_h = 1; L.dil_w = 1; L.act = act;
  std::vector<float> hw((size_t)Cout * Cin * 9), hb((size_t)Cout);
  cudaMemcpyAsync(hw.data(), wgt, hw.size() * sizeof(float), cudaMemcpyDeviceToHost, s);
  cudaMemcpyAsync(hb.data(), bias, hb.size() * sizeof(float), cudaMemcpyDeviceToHost, s);
  cudaStreamSynchronize(s);
  L.w_host.assign((size_t)9 * L.CinPad * L.CoutPad, 0.f);
  L.bias_host.assign((size_t)L.CoutPad, 0.f);
  for (int co = 0; co < Cout; ++co) {
    L.bias_host[(size_t)co] = hb[(size_t)co];
    for (int ci = 0; ci < Cin; ++ci) {
      const int pc = ci < Cl ? ci : cl_pad + (ci - Cl);   // packed position: [up Cl | pad | skip Cs]
      for (int t = 0; t < 9; ++t)
        L.w_host[((size_t)t * L.CinPad + pc) * L.CoutPad + co] = hw[((size_t)co * Cin + ci) * 9 + t];
    }
  }
  L.w = (float*)dalloc(L.w_host.size() * sizeof(float));
  L.bias = (float*)dalloc(L.bias_host.size() * sizeof(float));
  bool ok = blow.hi && bcat.hi && bout.hi && L.w && L.bias;
  if (ok) {
    cudaMemcpy(L.w, L.w_host.data(), L.w_host.size() * sizeof(float), cudaMemcpyHostToDevice);
    cudaMemcpy(L.bias, L.bias_host.data(), L.bias_host.size() * sizeof(float), cudaMemcpyHostToDevice);
    ok = ck(launch_nchw_to_act(low_nchw, Cl, blow.all(N), s), "nchw_to_act low") &&
         ck(launch_nchw_to_act(skip_nchw, Cs, bcat.view(N, 0, H, cl_pad, cin_pad - cl_pad), s), "nchw_to_act skip");
  }
  if (ok) ok = tc_prepare(L, err, allocs_);
  const int saved_mode = cfg_.conv_mode, saved_fuse = g_tc_debug[5];
  cfg_.conv_mode = 0;
  g_tc_debug[5] = fused ? 1 : 0;
  if (ok && fused && !tc_can_fuse_upsample(L, bcat.all(N), bout.view(N, 0, H, 0, Cout), blow.all(N))) {
    err = "debug_decoder: geometry not supported by the fused row kernel";
    ok = false;
  }
  if (ok) ok = run_decoder(L, blow.all(N), bcat, N, bout.view(N, 0, H, 0, Cout), s);
  cfg_.conv_mode = saved_mode;
  g_tc_debug[5] = saved_fuse;
  if (ok) ok = ck(launch_act_to_nchw(bout.view(N, 0, H, 0, Cout), Cout, y_nchw, s), "act_to_nchw");
  if (ok) ok = ck(cudaStreamSynchronize(s), "debug_decoder sync");
  L.tc.reset();
  for (void* p : allocs_) cudaFree(p);
  allocs_.clear();
  std::swap(tmp, allocs_);
  return ok;
}

bool Engine::debug_read(const char* what, float* out, int64_t cap, int64_t* dims, cudaStream_t s) {
  cudaSetDevice(cfg_.device);
  const std::string w(what);
  const int N = last_n_;
  const int nout = cfg_.nout, max_bin = cfg_.n_fft / 2;
  ActView v;
  int C = 0;
  if (w == "f3") { v = f3_.all(N); C = nout; }
  else if (w == "aux1") { v = in3_.view(N, 0, max_bin, pos_aux1_, nout / 4); C = nout / 4; }
  else if (w == "aux2") { v = in3_.view(N, 0, max_bin, pos_aux2_, nout / 2); C = nout / 2; }
  else if (w == "x") { v = in3_.view(N, 0, max_bin, pos_x_, 2); C = 2; }
  else if (w == "o1") { v = o1_.all(N); C = o1_.C; }
  else if (w == "o2") { v = o2_.all(N); C = o2_.C; }
  else {
    // "<net index>.<buffer>" e.g. "4.e5", "0.d2"
    int ni = w.size() > 2 && w[1] == '.' ? w[0] - '0' : -1;
    if (ni < 0 || ni > 4) { err = "debug_read: unknown tensor " + w; return false; }
    BaseNetPlan& P = nets_[ni];
    const std::string b = w.substr(2);
    // the LSTM branch's fp32 planes, copied raw; dims are their LstmPlan layout padded with 1s
    const LstmPlan& Q = P.lstm;
    const float* plane = nullptr;
    int64_t pd[4] = {0, 0, 0, 1};
    if (b == "lstm_l0") { plane = Q.l0; pd[0] = N; pd[1] = Q.bins; pd[2] = Q.T; }
    else if (b == "lstm_xp") { plane = Q.xp; pd[0] = N; pd[1] = Q.T; pd[2] = 8 * Q.hid; }
    else if (b == "lstm_hs") { plane = Q.hs; pd[0] = N; pd[1] = Q.T; pd[2] = 2 * Q.hid; }
    else if (b == "lstm_y") { plane = Q.y; pd[0] = Q.bins; pd[1] = N; pd[2] = Q.T; }
    if (plane) {
      const int64_t count = pd[0] * pd[1] * pd[2];
      for (int i = 0; i < 4; ++i) dims[i] = pd[i];
      if (count > cap) { err = "debug_read: output buffer too small"; return false; }
      return ck(cudaMemcpyAsync(out, plane, sizeof(float) * (size_t)count, cudaMemcpyDeviceToDevice, s), "debug_read");
    }
    const Buffer* buf = nullptr;
    if (b == "cat1") buf = &P.cat1; else if (b == "cat2") buf = &P.cat2; else if (b == "cat3") buf = &P.cat3;
    else if (b == "cat4") buf = &P.cat4; else if (b == "e5") buf = &P.e5; else if (b == "acat") buf = &P.acat;
    else if (b == "ao") buf = &P.ao; else if (b == "d4") buf = &P.d4; else if (b == "d3") buf = &P.d3;
    else if (b == "d2") buf = &P.d2; else if (b == "t2") buf = &P.t2; else if (b == "f1") buf = &P.f1;
    else if (b == "t3") buf = &P.t3; else if (b == "t4") buf = &P.t4; else if (b == "t5") buf = &P.t5;
    else if (b == "pool") buf = &P.pool;
    else if (b == "lstm_up") {
      if (!P.lstm_own) { err = "debug_read: " + P.prefix + " keeps its up-sampled LSTM channel in cat1, not lstm_up"; return false; }
      buf = &P.lstm_up;
    }
    else { err = "debug_read: unknown buffer " + b; return false; }
    v = buf->all(N); C = buf->C;
  }
  const int64_t total = (int64_t)N * C * v.H * v.W;
  dims[0] = N; dims[1] = C; dims[2] = v.H; dims[3] = v.W;
  if (total > cap) { err = "debug_read: output buffer too small"; return false; }
  return ck(launch_act_to_nchw(v, C, out, s), "debug_read");
}

}  // namespace vr
