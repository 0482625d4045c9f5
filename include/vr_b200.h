/* vr_b200.h - C ABI of the B200-native vocal-remover inference hot path (libvr_b200.so).
 *
 * The reference (tsurumeso/vocal-remover @ 99f92fe) is pure Python and has NO plugin / FFI interface;
 * the drop-in boundary is the Python call surface used by inference.py:130-176 and pseudo.py:32-67.
 * Each entry point below names the reference call it replaces.  The Python mirror that binds these
 * with ctypes lives in vocal-remover_b200/lib/_native.py (see INTEGRATION.md).
 *
 * Conventions: plain pointers and sizes only (no torch types); every function returns 0 on success and a
 * negative value on error, with the message available from vr_last_error(); `stream` is a cudaStream_t
 * passed as void* (NULL = legacy default stream); unless stated otherwise pointers are DEVICE pointers on
 * the context's GPU and calls are asynchronous on `stream`.  A context is bound to one GPU and is not
 * thread-safe.  There is no CPU path: vr_create fails if no CUDA device is present.
 *
 * Array layouts are the reference's (row-major / C order):
 *   wave  float32    [2][L]
 *   spec  complex64  [2][bins][T]        bins = n_fft/2+1, T = 1 + L/hop       (lib/spec_utils.py:26-31)
 *   mask  float32    [2][bins][T]
 *   mag   float32    [N][2][bins][W]     W = cropsize                          (lib/nets.py:124)
 */
#ifndef VR_B200_H_
#define VR_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define VR_API __attribute__((visibility("default")))
#else
#define VR_API
#endif

typedef struct vr_ctx vr_ctx;

typedef struct vr_config {
  int32_t device;      /* CUDA device ordinal                                   (inference.py:124-129)  */
  int32_t n_fft;       /* --n_fft, power of two in [64, 4096]                    (inference.py:113)      */
  int32_t hop_length;  /* --hop_length                                           (inference.py:114)      */
  int32_t nout;        /* CascadedNet nout (32)                                  (inference.py:130)      */
  int32_t nout_lstm;   /* CascadedNet nout_lstm (128)                            (inference.py:130)      */
  int32_t cropsize;    /* --cropsize, multiple of 16, > 128                      (inference.py:116)      */
  int32_t max_batch;   /* windows per forward launch sequence (--batchsize)      (inference.py:115)      */
  int32_t conv_mode;   /* 0 = tcgen05 tensor-core conv where the tile fits, 1 = CUDA-core conv only     */
} vr_config;

/* nets.CascadedNet(n_fft, hop, nout, nout_lstm).to(device)                      (lib/nets.py:46-80)     */
VR_API int vr_create(const vr_config* cfg, vr_ctx** out);
VR_API void vr_destroy(vr_ctx* ctx);
/* Message of the last failed call on ctx (ctx may be NULL for a failed vr_create). */
VR_API const char* vr_last_error(const vr_ctx* ctx);

/* model.load_state_dict(...) (inference.py:131): one call per state_dict entry with its PyTorch key,
 * HOST pointer; dtype 0 = float32, 1 = int64.  vr_finalize_weights is strict (missing / unexpected key or
 * shape mismatch -> error), folds eval-mode BatchNorm into the convolutions and packs for the kernels.  */
VR_API int vr_load_tensor(vr_ctx* ctx, const char* name, int32_t dtype, int32_t ndim, const int64_t* shape,
                   const void* host_data);
VR_API int vr_finalize_weights(vr_ctx* ctx);

/* spec_utils.wave_to_spectrogram(wave, hop, n_fft) (lib/spec_utils.py:26-31).  absmax (device float*,
 * may be NULL) receives max|spec| = the normaliser of inference.py:74.                                  */
VR_API int vr_stft(vr_ctx* ctx, const float* wave, int64_t L, void* spec, int64_t T, float* absmax, void* stream);

/* spec_utils.spectrogram_to_wave(spec, hop) (lib/spec_utils.py:157-165): wave [2][hop*(T-1)].           */
VR_API int vr_istft(vr_ctx* ctx, const void* spec, int64_t T, float* wave, void* stream);

/* model.predict_mask(x) (lib/nets.py:124-131): mag [N][2][bins][W] -> mask [N][2][bins][W-2*64].        */
VR_API int vr_predict_mask(vr_ctx* ctx, const float* mag, int32_t N, float* mask, void* stream);

/* model.forward(x) / model(x) (lib/nets.py:82-117): the un-cropped mask [N][2][bins][W].                */
VR_API int vr_forward(vr_ctx* ctx, const float* mag, int32_t N, float* mask, void* stream);

/* norm_mode 0: max|spec| (Separator.separate, inference.py:74); 1: |lexicographic complex max| as numpy's
 * complex .max() gives in Separator.separate_tta (inference.py:87,94).  out = device float*.            */
VR_API int vr_normaliser(vr_ctx* ctx, const void* spec, int64_t T, int32_t norm_mode, float* out, void* stream);

/* Separator._separate over a shard of windows (inference.py:42-68): windows [first_window,
 * first_window+n_windows) of the spectrogram padded by pad_l zeros on the left, normalised by *norm
 * (device), are run through the net; mask frame j of the concatenated result is written to
 * mask[:, :, j - frame_shift] if that lies in [0, mask_T).  accumulate=1 averages with what is there
 * ((old+new)/2, the TTA combine of inference.py:98).  `mask` may be a peer-mapped pointer on another GPU
 * (multi-GPU gather written by the epilogue kernel itself over NVLink).                                 */
VR_API int vr_separate_windows(vr_ctx* ctx, const void* spec, int64_t T, const float* norm, int32_t pad_l,
                        int32_t first_window, int32_t n_windows, float* mask, int64_t mask_T,
                        int64_t frame_shift, int32_t accumulate, void* stream);

/* Mask of Separator.separate (tta=0, inference.py:70-77) / separate_tta (tta=1, inference.py:83-98).    */
VR_API int vr_separate(vr_ctx* ctx, const void* spec, int64_t T, int32_t tta, float* mask, void* stream);

/* Separator._postprocess without --postprocess (inference.py:32-36): y = mask*spec, v = (1-mask)*spec.  */
VR_API int vr_apply_mask(vr_ctx* ctx, const void* spec, const float* mask, int64_t T, void* y_spec, void* v_spec,
                  void* stream);

/* --postprocess / spec_utils.merge_artifacts (lib/spec_utils.py:60-93, inference.py:27-30) without moving the mask
 * off the device: frame_min[t] = min over (channel, bin) of mask[:, :, t] (device float[T]); the caller finds the
 * long above-threshold runs on the host from those T floats (lib/spec_utils.py:artifact_weights) and hands back one
 * fade weight per frame, which vr_mask_apply_weight applies in place: mask += weight[t] * (1 - mask).           */
VR_API int vr_mask_frame_min(vr_ctx* ctx, const float* mask, int64_t T, float* frame_min, void* stream);
VR_API int vr_mask_apply_weight(vr_ctx* ctx, float* mask, int64_t T, const float* weight, void* stream);

/* y/v waves straight from spec and mask: _postprocess + 2x spectrogram_to_wave fused
 * (inference.py:32-36,171,176).  wave_inst / wave_voc: [2][hop*(T-1)].                                 */
VR_API int vr_apply_mask_istft(vr_ctx* ctx, const void* spec, const float* mask, int64_t T, float* wave_inst,
                        float* wave_voc, void* stream);

/* Shard-sized pieces of the three calls above for the multi-GPU path (lib/distributed.py): the STFT of frames
 * [t0, t1) only, max|spec| over those frames (ranks all-reduce it to the normaliser of inference.py:74), and the
 * masked inverse STFT of output hops [k0, k1) = samples [hop*k0, hop*k1) of wave_inst / wave_voc [2][hop*(T-1)],
 * which may be peer-mapped buffers on another GPU (the overlap-add kernel then stores over NVLink).
 * spec / mask are the full-size [2][bins][T] arrays; only the columns the range touches are read / written.  */
VR_API int vr_stft_range(vr_ctx* ctx, const float* wave, int64_t L, void* spec, int64_t T, int64_t t0, int64_t t1,
                  void* stream);
VR_API int vr_normaliser_range(vr_ctx* ctx, const void* spec, int64_t T, int64_t t0, int64_t t1, float* out,
                        void* stream);
VR_API int vr_apply_mask_istft_range(vr_ctx* ctx, const void* spec, const float* mask, int64_t T, int64_t k0,
                              int64_t k1, float* wave_inst, float* wave_voc, void* stream);

/* Whole hot path with everything resident in HBM (inference.py:147-176 minus file I/O).                 */
VR_API int vr_separate_wave(vr_ctx* ctx, const float* wave, int64_t L, int32_t tta, float* wave_inst,
                     float* wave_voc, void* stream);

/* Same with HOST buffers (pinned recommended); copies in, runs, copies out and synchronises.            */
VR_API int vr_separate_wave_host(vr_ctx* ctx, const float* wave_host, int64_t L, int32_t tta, float* inst_host,
                          float* voc_host, void* stream);

/* Several tracks per call (not a reference surface: the reference separates one file per run).  A track is cut into
 * cropsize windows as in vr_separate; here the windows of ALL tracks share the forward batches of max_batch windows, so
 * short tracks and the last partial batch of each track do not each pay for a nearly empty forward.  Windows are
 * independent inside the net, and each track keeps its own normaliser and padding, so every mask equals the one
 * vr_separate gives for that track alone.  Every argument is checked before anything is launched; an error names the
 * offending track.
 *
 * vr_separate_many: Separator.separate / separate_tta (tta as in vr_separate) over n_tracks >= 1 tracks.  specs[i] is
 * a complex64 [2][bins][T[i]] spectrogram (T[i] >= 1), masks[i] receives the float32 [2][bins][T[i]] mask.  specs, T and
 * masks are HOST arrays of n_tracks entries; the pointers in specs and masks are DEVICE pointers.                   */
VR_API int vr_separate_many(vr_ctx* ctx, int32_t n_tracks, const void* const* specs, const int64_t* T, int32_t tta,
                            float* const* masks, void* stream);
/* vr_separate_wave over n_tracks >= 1 tracks: waves[i] float32 [2][L[i]] (L[i] >= 0) -> inst[i], voc[i]
 * [2][hop*(T_i-1)], T_i = 1 + L[i]/hop.  waves, L, inst and voc are HOST arrays of n_tracks entries holding DEVICE
 * pointers.  The STFT, the normalisers and the masked inverse STFT of all tracks are one launch each; the
 * workspaces grow with the total frame count of the call.                                                         */
VR_API int vr_separate_waves(vr_ctx* ctx, int32_t n_tracks, const float* const* waves, const int64_t* L, int32_t tta,
                             float* const* inst, float* const* voc, void* stream);

/* The sample-rate conversion inside librosa.load(path, sr=args.sr, res_type='kaiser_fast') (inference.py:136-138,
 * pseudo.py:47-50) = resampy.resample(y, orig_sr, sr, filter='kaiser_fast'): x [channels][n_in] -> y [channels][n_out],
 * n_out = (int64)(n_in * sample_ratio), sample_ratio = sr / orig_sr.  win / delta: DEVICE float64 arrays of nwin entries -
 * the half filter table (already multiplied by sample_ratio when it is < 1) and its first difference - with
 * table_per_crossing entries per zero crossing, as resampy.core.resample prepares them (lib/audio_io.py builds the
 * documented kaiser_fast table; a table taken from an installed resampy can be passed instead).  ctx may be NULL
 * (audio is loaded before a model exists): the call then runs on the calling thread's current device and its error
 * message is read with vr_last_error(NULL).  SURVEY 8(f) rank 2.                                            */
VR_API int vr_resample(vr_ctx* ctx, const float* x, int32_t channels, int64_t n_in, float* y, int64_t n_out,
                       double sample_ratio, const double* win, const double* delta, int32_t nwin,
                       int32_t table_per_crossing, void* stream);

/* Multi-GPU mask exchange over NVLink peer memory (one process per GPU).  The owner (rank 0) allocates the
 * whole-track mask with vr_shared_alloc and publishes the 64-byte CUDA IPC handle; every other rank maps it
 * with vr_shared_open and passes the mapped pointer as `mask` to vr_separate_windows, so the mask epilogue
 * kernel itself stores its shard into rank 0's HBM - the "gather" of Separator._separate's concatenate
 * (inference.py:63-66) fused into the producing kernel.  vr_shared_close unmaps (owner=0) or frees (owner=1). */
VR_API int vr_shared_alloc(vr_ctx* ctx, int64_t bytes, void** dev_ptr, unsigned char* handle64);
VR_API int vr_shared_open(vr_ctx* ctx, const unsigned char* handle64, void** dev_ptr);
VR_API int vr_shared_close(vr_ctx* ctx, void* dev_ptr, int32_t owner);

/* Number of kernels launched by this context so far (bench.py 'gpu_launches').                           */
VR_API int64_t vr_launch_count(const vr_ctx* ctx);

/* CUDA-event timing of every convolution launch between enable(1) and read (bench.py roofline):
 * out[0..2] = tensor-core conv {ms, algorithmic FLOPs, launches}, out[3..5] = CUDA-core conv likewise.    */
VR_API int vr_profile_enable(vr_ctx* ctx, int32_t on);
VR_API int vr_profile_read(vr_ctx* ctx, double* out6);
/* Per-launch detail of the same records as text, one line per convolution launch in launch order:
 * "<state_dict prefix of the layer>[+up] N Hout Wout tensor_core(0/1) ms gflop".  Writes at most cap bytes
 * (NUL-terminated) and stores the size needed in *needed (either may be NULL / 0 to query).                */
VR_API int vr_profile_dump(vr_ctx* ctx, char* text, int64_t cap, int64_t* needed);

/* ---- validation hooks used by tests/ (not part of the reference surface) ---------------------------- */
/* One Conv2DBNActiv-shaped layer (lib/layers.py:8-26; BN already folded into w/bias by the caller):
 * x [N][Cin][H][W] -> y [N][Cout][Ho][Wo]; use_tc selects the tcgen05 kernel (error if tile does not fit). */
VR_API int vr_debug_conv(vr_ctx* ctx, const float* x, int32_t N, int32_t Cin, int32_t H, int32_t W, const float* w,
                  const float* bias, int32_t Cout, int32_t k, int32_t stride, int32_t dil_h, int32_t dil_w,
                  int32_t act, int32_t use_tc, float* y, void* stream);
/* One Decoder-shaped layer (lib/layers.py:51-64, BN folded by the caller): low [N][Cl][h][w] is bilinearly
 * upsampled x2 (align_corners=True), concatenated with skip [N][Cs][2h][2w] and convolved 3x3 -> y [N][Cout][2h][2w];
 * fused = 1 runs the upsample inside the row-streaming tensor-core kernel, 0 as a separate kernel.              */
VR_API int vr_debug_decoder(vr_ctx* ctx, const float* low, int32_t N, int32_t Cl, int32_t h, int32_t w, const float* skip,
                     int32_t Cs, const float* wgt, const float* bias, int32_t Cout, int32_t act, int32_t fused, float* y,
                     void* stream);
/* Process-wide debug knobs of the tensor-core kernels (keys 0..7): key 0 = 1 records the row-streaming kernel's
 * timeline for vr_debug_trace (builds with -DVR_TRACE), key 1 = 1 disables that kernel, key 2 = 1 makes vr_debug_conv use the row kernel's
 * 64-output-channel tile, key 4 = k sets the number of interpolation slots of the fused upsample, key 5 = 1 (default)
 * fuses the decoder upsample into the row-streaming kernel and lets vr_create choose the fused dec1 layouts (0: staged
 * layout everywhere; set before vr_create), key 6 = 1 (default) skips 8-channel input groups whose weights are all
 * zero.                                                                                                        */
VR_API int vr_debug_set(int32_t key, int32_t value);
/* timeline of CTA 0 of the last row-kernel launch made with vr_debug_set(0, 1): 3 roles x 2048 events x 3 clock64 stamps
 * (MMA issuer / TMA producer / interpolation warp 0), copied to HOST memory; returns the number of values or -1 */
VR_API int64_t vr_debug_trace(uint64_t* host_out, int64_t capacity);
/* Internal tensor of the last forward, copied to the DEVICE buffer out (capacity floats); dims receives 4 sizes.
 * Activations (split-bf16 buffers, returned as hi + lo in float32 NCHW, every channel of the buffer incl. padding;
 * dims = [N, C, H, W]):
 *   "x", "aux1", "aux2"        slots of the stage input buffer, all max_bin rows ([0, bins/2) low band, rest high band)
 *   "o1", "o2"                 stage-1 / stage-2 low-band BaseNet outputs before the 1x1 bridges
 *   "f3"                       stage-3 output
 *   "<k>.<buf>"                buffer of BaseNet k (0 stg1_low, 1 stg1_high, 2 stg2_low, 3 stg2_high, 4 stg3_full):
 *                              cat1 cat2 cat3 cat4 (decoder concat inputs), t2 t3 t4 t5 (encoder conv1 outputs),
 *                              e5, pool (ASPP frequency mean), f1, acat, ao, d4, d3, d2, and lstm_up (only for nets that
 *                              keep the up-sampled LSTM channel in a buffer of its own; an error otherwise)
 * LSTM branch fp32 planes of BaseNet k, copied raw (dims = the layout padded with 1s):
 *   "<k>.lstm_l0"  [N, bins, T, 1]      1x1 input convolution, pre-activation sums
 *   "<k>.lstm_xp"  [N, T, 8*hid, 1]     gate pre-activations, forward then reverse direction
 *   "<k>.lstm_hs"  [N, T, 2*hid, 1]     hidden states, forward then reverse direction
 *   "<k>.lstm_y"   [bins, N, T, 1]      dense + BatchNorm1d + ReLU output                                      */
VR_API int vr_debug_read(vr_ctx* ctx, const char* what, float* out, int64_t capacity, int64_t* dims, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VR_B200_H_ */
