// Host-side launch prototypes for the hand-written sm_100a kernels of the hot path.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "common.cuh"

namespace vr {

// ---- convolution (conv_simt.cu / conv_tc.cu) -------------------------------------------------
cudaError_t launch_conv_simt(const ConvParams& p, cudaStream_t stream);

// ---- bandwidth kernels (elementwise.cu) ------------------------------------------------------
// |X|/norm of window g = first_window + n, frame tw -> dst channels [0,2) ; spec is complex64 [2][bins][T]
cudaError_t launch_pack_mag_from_spec(const float2* spec, int bins, int64_t T, int max_bin, int W, int roi,
                                      int pad_l, int first_window, const float* norm, ActView dst,
                                      cudaStream_t stream);
// mag is float32 NCHW [N][2][bins][W] (the reference predict_mask input, lib/nets.py:124)
cudaError_t launch_pack_mag_from_float(const float* mag, int bins, int max_bin, ActView dst, cudaStream_t stream);
cudaError_t launch_nchw_to_act(const float* x, int C, ActView dst, cudaStream_t stream);
cudaError_t launch_act_to_nchw(ActView src, int C, float* y, cudaStream_t stream);
cudaError_t launch_upsample2x(ActView in, ActView out, cudaStream_t stream);
// fp32 plane in[(n) in_sn][(row) in_sh][col] (inH x inW per image) -> channel 0 of the 16- or 8-channel group `out`
// (the other channels written as zeros), same interpolation arithmetic as launch_upsample2x
cudaError_t launch_upsample2x_c1(const float* in, int inH, int inW, int64_t in_sn, int64_t in_sh, ActView out,
                                 cudaStream_t stream);
cudaError_t launch_pool_freq_mean(ActView in, ActView out, cudaStream_t stream);
cudaError_t launch_broadcast_rows(ActView in, ActView out, cudaStream_t stream);

struct MaskOutParams {
  ActView f3;          // (N, max_bin, W, nout)
  const float* w;      // [2][nout]  (CascadedNet.out.weight, lib/nets.py:79)
  float* out;
  int64_t stride_n, stride_c, stride_bin;  // element strides of the destination; frames are contiguous
  int offset;          // model.offset (64): frames [offset, W-offset) are kept (lib/nets.py:127-129)
  int64_t t_base0;     // destination frame index of frame `offset` of window 0, before stride_n is applied
  int64_t t_limit;     // frames with (t_base0 + n*roi_t + tw-offset) outside [0, t_limit) are dropped
  int roi_t;           // per-window frame advance used only for the limit test
  int accumulate;      // 1: out = (out + mask) * 0.5  (TTA average, inference.py:98)
};
cudaError_t launch_mask_out(const MaskOutParams& p, cudaStream_t stream);

// ---- several tracks per launch (vr_separate_many / vr_separate_waves) -----------------------------------------
// One window of a packed forward batch: batch slot n reads wins[n].  Pack: |X|/norms[norm] of window `window` of the
// spectrogram spec [2][bins][T] padded by pad_l zeros on the left.  Mask epilogue: kept frame tr of the window goes to
// mask[c][bin][t_base + tr] (mask [2][bins][T]) if that lies in [0, T); accumulate = 1 averages with what is there.
struct WinDesc {
  const float2* spec;
  float* mask;
  int64_t T;
  int64_t t_base;
  int pad_l, window, norm, accumulate;
};
cudaError_t launch_pack_mag_many(const WinDesc* wins, int bins, int max_bin, int W, int roi, const float* norms,
                                 ActView dst, cudaStream_t stream);
cudaError_t launch_mask_out_many(ActView f3, const float* w, int offset, const WinDesc* wins, cudaStream_t stream);
// normaliser of each track: spec with n complex elements -> out[track]
struct NormTrack {
  const float2* spec;
  int64_t n;
};
// mode 0: max|X| (launch_absmax), 1: |lexicographic max| with the zero padding taking part (launch_lexmax_abs);
// scratch: n_tracks entries; max_n: largest n of the table (sizes the grid)
cudaError_t launch_normaliser_many(const NormTrack* tracks, int n_tracks, int64_t max_n, int mode,
                                   unsigned long long* scratch, float* out, cudaStream_t stream);

cudaError_t launch_absmax(const float2* spec, int64_t n, float* out_absmax, cudaStream_t stream);
// max |spec[r][t]| over rows r < nrows and frames t in [t0, t1) of a [nrows][T] array
cudaError_t launch_absmax_range(const float2* spec, int nrows, int64_t T, int64_t t0, int64_t t1, float* out_absmax,
                                cudaStream_t stream);
cudaError_t launch_lexmax_abs(const float2* spec, int64_t n, unsigned long long* scratch, float* out_norm,
                              cudaStream_t stream);
cudaError_t launch_mask_frame_min(const float* mask, int rows, int64_t T, float* out, cudaStream_t stream);
cudaError_t launch_mask_apply_weight(float* mask, int rows, int64_t T, const float* weight, cudaStream_t stream);
cudaError_t launch_apply_mask(const float2* spec, const float* mask, int64_t n, float2* y, float2* v,
                              cudaStream_t stream);

// ---- LSTM branch (lstm.cu), reference lib/layers.py:108-133 ------------------------------------
// 1x1 conv (C -> 1), pre-activation sums as an fp32 plane l0[n][bin][t] (the row kernel's epilogue accumulates the same
// sums when the layer that produces `in` runs there: RowsDot in tc_plan.h)
cudaError_t launch_lstm_inconv(ActView in, const float* w, float* l0, cudaStream_t stream);
// xp[(n,t)][gates] = relu(l0[n][:][t] + conv_bias) . wih[gates][:]^T + bih   (gates = 8 * hid)
cudaError_t launch_lstm_input_projection(const float* l0, float conv_bias, const float* wih, const float* bih, float* xp,
                                         int N, int T, int bins, int gates, cudaStream_t stream);
// xp: [n][t][2][4*hid] gate pre-activations (input projection + both biases), whh: [2][4*hid][hid]
// hs: [n][t][2*hid]
cudaError_t launch_lstm_recurrence(const float* xp, const float* whh, float* hs, int N, int T, int hid,
                                   cudaStream_t stream);
// y[bin][(n,t)] = relu(scale[bin] * (wd[bin][:] . hs[(n,t)][:]) + shift[bin]),  wd: [bins][K], NT = N * T
cudaError_t launch_lstm_dense(const float* hs, const float* wd, const float* scale, const float* shift, int NT, int K,
                              int bins, float* y, cudaStream_t stream);
// y[bin][n][t] -> channel `ch` of dst[n][bin][t][.] (split bf16)
cudaError_t launch_lstm_plane_to_channel(const float* y, int N, int T, int bins, ActView dst, int ch,
                                         cudaStream_t stream);

// ---- STFT / iSTFT (fft.cu), reference lib/spec_utils.py:26-31,157-165 (librosa semantics, SURVEY App. A)
// frames [t0, t1) only (the full-track call is t0 = 0, t1 = T)
cudaError_t launch_stft(const float* wave, int64_t L, int n_fft, int hop, float2* spec, int64_t T, int64_t t0,
                        int64_t t1, const float2* twiddle, const float* window, cudaStream_t stream);
// frames_a[c][t][:] = hann * irfft(spec * mask), frames_b = hann * irfft(spec * (1 - mask));
// mask == nullptr: frames_a = hann * irfft(spec), frames_b unused
// frames [t_first, t_first + nfr) of the track into a scratch laid out [c][nfr][n_fft]
cudaError_t launch_istft_frames(const float2* spec, const float* mask, int n_fft, int64_t T, int64_t t_first,
                                int64_t nfr, float* frames_a, float* frames_b, const float2* twiddle,
                                const float* window, cudaStream_t stream);
// overlap-add + window-sum-square normalisation + centre trim of output samples [s0, s1) of wave [2][hop*(T-1)]
cudaError_t launch_istft_ola(const float* frames_a, const float* frames_b, int n_fft, int hop, int64_t T,
                             int64_t t_first, int64_t nfr, int64_t s0, int64_t s1, float* wave_a, float* wave_b,
                             const float* window, cudaStream_t stream);

// Ragged forms over several tracks, one launch each.  A track's CTAs (STFT, iSTFT frames: cta0) and its output samples
// (overlap-add: s0, 2 * hop * (T-1) per track) start at prefix sums of the earlier tracks' counts, ascending; a CTA or
// thread finds its track by binary search.  The iSTFT frames of track i sit at frames_a / frames_b + 2 * frame_off *
// n_fft, laid out [c][T][n_fft] as launch_istft_frames writes them.
struct FftTrack {
  const float* wave;   // STFT input [2][L]
  float2* spec;        // [2][bins][T] (iSTFT: read)
  const float* mask;   // iSTFT: [2][bins][T]
  float* wave_a;       // iSTFT outputs [2][hop*(T-1)]
  float* wave_b;
  int64_t L, T;
  int64_t frame_off;   // sum of the earlier tracks' T
  int64_t cta0;        // first CTA of the track in launch_stft_many / launch_istft_frames_many
  int64_t s0;          // first output sample of the track in launch_istft_ola_many
};
// CTAs a track of T frames takes in launch_stft_many / launch_istft_frames_many (the same count for both)
int64_t fft_ctas_per_track(int n_fft, int64_t T);
cudaError_t launch_stft_many(const FftTrack* tracks, int n_tracks, int64_t total_ctas, int n_fft, int hop,
                             const float2* twiddle, const float* window, cudaStream_t stream);
cudaError_t launch_istft_frames_many(const FftTrack* tracks, int n_tracks, int64_t total_ctas, int n_fft, float* frames_a,
                                     float* frames_b, const float2* twiddle, const float* window, cudaStream_t stream);
cudaError_t launch_istft_ola_many(const FftTrack* tracks, int n_tracks, int64_t total_samples, int n_fft, int hop,
                                  const float* frames_a, const float* frames_b, const float* window, cudaStream_t stream);

// ---- sample-rate conversion (resample.cu), resampy.resample(filter='kaiser_fast') behind librosa.load ----------
// x [C][n_in] -> y [C][n_out], n_out = int(n_in * sample_ratio); win / delta: the (ratio-scaled) half filter table and
// its first difference, nwin entries, num_table entries per zero crossing (oracle/resample_oracle.py: prepare)
cudaError_t launch_resample_sinc(const float* x, int C, int64_t n_in, float* y, int64_t n_out, double sample_ratio,
                                 const double* win, const double* delta, int nwin, int num_table, cudaStream_t stream);

}  // namespace vr
