// Framed Hann-windowed STFT and window-sum-square-normalised overlap-add inverse STFT.
//
// Device replacement for the reference's two librosa calls (lib/spec_utils.py:26-31 and 157-165;
// librosa 0.10 semantics restated in SURVEY.md App. A and oracle/stft_oracle.py):
//   stft : zero centre padding n_fft/2, frame t = y_p[t*hop : t*hop+n_fft], periodic Hann, rfft
//          -> complex64 [2][n_fft/2+1][T], T = 1 + L/hop
//   istft: irfft(1/N) * Hann, overlap-add at hop, / sum(Hann^2) where > tiny, trim n_fft/2 both ends
// One CTA transforms one frame with a shared-memory radix-2 FFT.  Two real signals ride in one
// complex transform: the stereo pair (L + iR) forward, the two stems (instruments + i*vocals)
// inverse, so the mask multiply of Separator._postprocess (inference.py:32-36) is fused into the
// inverse transform's load.
#include "common.cuh"
#include "kernels.h"

namespace vr {

__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
  return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}

// In-place radix-2 DIT on bit-reversed data in shared memory.  tw[q] = exp(-2 pi i q / NF), q < NF/2.
// INVERSE uses conj(tw).
template <bool INVERSE>
__device__ __forceinline__ void fft_inplace(float2* z, const float2* __restrict__ tw, int NF, int logn) {
  for (int s = 1; s <= logn; ++s) {
    const int half = 1 << (s - 1);
    const int tstep = NF >> s;
    for (int k = threadIdx.x; k < (NF >> 1); k += blockDim.x) {
      const int j = k & (half - 1);
      const int i0 = ((k >> (s - 1)) << s) + j;
      const int i1 = i0 + half;
      float2 w = __ldg(tw + j * tstep);
      if (INVERSE) w.y = -w.y;
      const float2 a = z[i0];
      const float2 b = cmul(z[i1], w);
      z[i0] = make_float2(a.x + b.x, a.y + b.y);
      z[i1] = make_float2(a.x - b.x, a.y - b.y);
    }
    __syncthreads();
  }
}

// frame t of the track, one CTA, z: NF float2 of shared memory
__device__ __forceinline__ void stft_frame(const float* __restrict__ wave, int64_t L, int NF, int logn, int hop,
                                           float2* __restrict__ spec, int64_t T, int64_t t,
                                           const float2* __restrict__ tw, const float* __restrict__ win, float2* z) {
  const int64_t s0 = t * hop - NF / 2;
  for (int n = threadIdx.x; n < NF; n += blockDim.x) {
    const int64_t s = s0 + n;
    float l = 0.f, r = 0.f;
    if (s >= 0 && s < L) {
      l = wave[s];
      r = wave[L + s];
    }
    const float w = win[n];
    z[__brev((unsigned)n) >> (32 - logn)] = make_float2(l * w, r * w);
  }
  __syncthreads();
  fft_inplace<false>(z, tw, NF, logn);
  const int bins = NF / 2 + 1;
  for (int k = threadIdx.x; k < bins; k += blockDim.x) {
    const float2 a = z[k];
    const float2 b = z[(NF - k) & (NF - 1)];
    spec[((int64_t)0 * bins + k) * T + t] = make_float2(0.5f * (a.x + b.x), 0.5f * (a.y - b.y));
    spec[((int64_t)1 * bins + k) * T + t] = make_float2(0.5f * (a.y + b.y), -0.5f * (a.x - b.x));
  }
}

__global__ void __launch_bounds__(256) stft_kernel(const float* __restrict__ wave, int64_t L, int NF, int logn,
                                                   int hop, float2* __restrict__ spec, int64_t T, int64_t t_first,
                                                   const float2* __restrict__ tw, const float* __restrict__ win) {
  extern __shared__ float2 z[];
  stft_frame(wave, L, NF, logn, hop, spec, T, t_first + blockIdx.x, tw, win, z);
}

// index of the track whose [first, next first) range holds x (tracks sorted by first, tracks[0].first == 0)
template <int64_t FftTrack::*FIRST>
__device__ __forceinline__ int find_track(const FftTrack* __restrict__ tracks, int n_tracks, int64_t x) {
  int lo = 0, hi = n_tracks - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (tracks[mid].*FIRST <= x) lo = mid; else hi = mid - 1;
  }
  return lo;
}


// ------------------------------------------------------------------------------------------------
// Fast path for n_fft = 2048: 2048 = 8 * 8 * 8 * 4.  Each of the 256 threads holds eight points in registers per pass
// (in-place decimation in frequency: three radix-8 passes and one radix-4 pass with four shared-memory exchanges, against
// eleven for the radix-2 kernel above), and one CTA transforms kFR consecutive frames between barriers, so that its
// spectrum accesses - the spectrogram is stored with the frame index contiguous - cover whole 32-byte sectors.
constexpr int kFR = 4;   // frames per CTA
constexpr int kF2048 = 2048;
// 4 points of padding per 32: the stride-32 accesses of pass 3 then hit distinct banks
__host__ __device__ constexpr int fpad(int i) { return i + ((i >> 5) << 2); }
constexpr int kFrameSlots = kF2048 + (kF2048 >> 5) * 4;   // 2304 float2 per frame buffer

__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ float2 mul_mi(float2 a) { return make_float2(a.y, -a.x); }   // a * (-i)

// forward 4-point DFT, natural order in and out
__device__ __forceinline__ void dft4(float2& x0, float2& x1, float2& x2, float2& x3) {
  const float2 s0 = cadd(x0, x2), s1 = csub(x0, x2), s2 = cadd(x1, x3), s3 = mul_mi(csub(x1, x3));
  x0 = cadd(s0, s2);
  x1 = cadd(s1, s3);
  x2 = csub(s0, s2);
  x3 = csub(s1, s3);
}

// forward 8-point DFT, natural order in and out
__device__ __forceinline__ void dft8(float2* a) {
  const float c = 0.70710678118654752440f;
  float2 b0 = cadd(a[0], a[4]), b1 = cadd(a[1], a[5]), b2 = cadd(a[2], a[6]), b3 = cadd(a[3], a[7]);
  float2 d0 = csub(a[0], a[4]), d1 = csub(a[1], a[5]), d2 = csub(a[2], a[6]), d3 = csub(a[3], a[7]);
  d1 = make_float2(c * (d1.x + d1.y), c * (d1.y - d1.x));    // * w8^1
  d2 = mul_mi(d2);                                           // * w8^2
  d3 = make_float2(c * (d3.y - d3.x), -c * (d3.x + d3.y));   // * w8^3
  dft4(b0, b1, b2, b3);   // X0 X2 X4 X6
  dft4(d0, d1, d2, d3);   // X1 X3 X5 X7
  a[0] = b0; a[2] = b1; a[4] = b2; a[6] = b3;
  a[1] = d0; a[3] = d1; a[5] = d2; a[7] = d3;
}

// exp(-2 pi i idx / 2048), idx in [0, 2048), from the half table tw[q] = exp(-2 pi i q / 2048), q < 1024
__device__ __forceinline__ float2 w2048(const float2* __restrict__ tw, int idx) {
  const float2 w = __ldg(tw + (idx & 1023));
  return (idx & 1024) ? make_float2(-w.x, -w.y) : w;
}

// One radix-8 pass over the kFR frame buffers: points base + step * r, r < 8, of every frame; output q is multiplied by
// w[q] and goes back to the slot of input q (in place: every thread owns its eight slots).
__device__ __forceinline__ void radix8_pass(float2* z, int base, int step, const float2* w) {
  float2 a[8];
#pragma unroll 1
  for (int f = 0; f < kFR; ++f) {
    float2* zf = z + f * kFrameSlots;
#pragma unroll
    for (int r = 0; r < 8; ++r) a[r] = zf[fpad(base + step * r)];
    dft8(a);
#pragma unroll
    for (int q = 1; q < 8; ++q) a[q] = cmul(a[q], w[q]);
#pragma unroll
    for (int q = 0; q < 8; ++q) zf[fpad(base + step * q)] = a[q];
  }
}

// In-place forward FFT of the kFR padded frame buffers z[f][fpad(n)]: natural order in, natural order out; ends with
// a barrier.  Index split n = n1 + 256 r (pass 1), then inside the sequence of output digit q1: n1 = n2 + 32 r (pass 2),
// inside (q1, q2): n2 = n3 + 4 r (pass 3), leaving 512 sequences of four points (pass 4).  X[q1 + 8 q2 + 64 q3 + 512 k4].
__device__ __forceinline__ void fft2048_frames(float2* z, const float2* __restrict__ tw) {
  const int t = threadIdx.x;
  float2 w[8];
  w[0] = make_float2(1.f, 0.f);
#pragma unroll
  for (int q = 1; q < 8; ++q) w[q] = w2048(tw, t * q);
  radix8_pass(z, t, 256, w);
  __syncthreads();
  {
    const int n2 = t & 31;
#pragma unroll
    for (int q = 1; q < 8; ++q) w[q] = w2048(tw, 8 * n2 * q);
    radix8_pass(z, (t >> 5) * 256 + n2, 32, w);
  }
  __syncthreads();
  {
    const int n3 = t & 3;
#pragma unroll
    for (int q = 1; q < 8; ++q) w[q] = w2048(tw, 64 * n3 * q);
    radix8_pass(z, (t >> 2) * 32 + n3, 4, w);
  }
  __syncthreads();
  // pass 4: sequence u = q3 + 8 q2 + 64 q1 sits at [4 u, 4 u + 4); thread t takes u = t and t + 256.  The results go
  // back to their natural slots once every thread has read its inputs.
#pragma unroll 1
  for (int f = 0; f < kFR; ++f) {
    float2* zf = z + f * kFrameSlots;
    float2 a[8];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int u = t + 256 * h;
#pragma unroll
      for (int r = 0; r < 4; ++r) a[4 * h + r] = zf[fpad(4 * u + r)];
      dft4(a[4 * h], a[4 * h + 1], a[4 * h + 2], a[4 * h + 3]);
    }
    __syncthreads();
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int u = t + 256 * h;
      const int k0 = (u >> 6) + 8 * ((u >> 3) & 7) + 64 * (u & 7);
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4) zf[fpad(k0 + 512 * k4)] = a[4 * h + k4];
    }
  }
  __syncthreads();
}

// frames [t0, min(t0 + kFR, t_end)) of the track, one CTA
__device__ __forceinline__ void stft2048_frames(const float* __restrict__ wave, int64_t L, int hop,
                                                float2* __restrict__ spec, int64_t T, int64_t t0, int64_t t_end,
                                                const float2* __restrict__ tw, const float* __restrict__ win, float2* z) {
  constexpr int NF = kF2048;
  for (int f = 0; f < kFR; ++f) {
    const int64_t s0 = (t0 + f) * hop - NF / 2;
    float2* zf = z + f * kFrameSlots;
    for (int n = threadIdx.x; n < NF; n += blockDim.x) {
      const int64_t s = s0 + n;
      float l = 0.f, r = 0.f;
      if (s >= 0 && s < L && t0 + f < t_end) {
        l = wave[s];
        r = wave[L + s];
      }
      const float w = win[n];
      zf[fpad(n)] = make_float2(l * w, r * w);
    }
  }
  __syncthreads();
  fft2048_frames(z, tw);
  constexpr int bins = NF / 2 + 1;
  const int nf = (int)(t_end - t0 < kFR ? t_end - t0 : kFR);
  for (int k = threadIdx.x; k < bins; k += blockDim.x) {
    float2 l[kFR], r[kFR];
#pragma unroll
    for (int f = 0; f < kFR; ++f) {
      const float2 a = z[f * kFrameSlots + fpad(k)];
      const float2 b = z[f * kFrameSlots + fpad((NF - k) & (NF - 1))];
      l[f] = make_float2(0.5f * (a.x + b.x), 0.5f * (a.y - b.y));
      r[f] = make_float2(0.5f * (a.y + b.y), -0.5f * (a.x - b.x));
    }
    float2* pl = spec + ((int64_t)0 * bins + k) * T + t0;
    float2* pr = spec + ((int64_t)1 * bins + k) * T + t0;
    if (nf == kFR && ((reinterpret_cast<uintptr_t>(pl) | reinterpret_cast<uintptr_t>(pr)) & 15) == 0) {
      reinterpret_cast<float4*>(pl)[0] = make_float4(l[0].x, l[0].y, l[1].x, l[1].y);
      reinterpret_cast<float4*>(pl)[1] = make_float4(l[2].x, l[2].y, l[3].x, l[3].y);
      reinterpret_cast<float4*>(pr)[0] = make_float4(r[0].x, r[0].y, r[1].x, r[1].y);
      reinterpret_cast<float4*>(pr)[1] = make_float4(r[2].x, r[2].y, r[3].x, r[3].y);
    } else {
#pragma unroll
      for (int f = 0; f < kFR; ++f)
        if (f < nf) {
          pl[f] = l[f];
          pr[f] = r[f];
        }
    }
  }
}

__global__ void __launch_bounds__(256) stft2048_kernel(const float* __restrict__ wave, int64_t L, int hop,
                                                       float2* __restrict__ spec, int64_t T, int64_t t_first, int64_t t_end,
                                                       const float2* __restrict__ tw, const float* __restrict__ win) {
  extern __shared__ float2 z[];
  stft2048_frames(wave, L, hop, spec, T, t_first + (int64_t)blockIdx.x * kFR, t_end, tw, win, z);
}

// Inverse transform through the forward one: ifft(x) = conj(fft(conj(x))).  Channel c, scratch frames
// [fr0, min(fr0 + kFR, nfr)) = track frames t_first + fr0 ..., one CTA.
__device__ __forceinline__ void istft2048_frames(const float2* __restrict__ spec, const float* __restrict__ mask,
                                                 int64_t T, int64_t t_first, int64_t nfr, int64_t fr0, int c,
                                                 float* __restrict__ frames_a, float* __restrict__ frames_b,
                                                 const float2* __restrict__ tw, const float* __restrict__ win,
                                                 float2* z) {
  constexpr int NF = kF2048;
  constexpr int bins = NF / 2 + 1;
  const int64_t t0 = t_first + fr0;
  const int nf = (int)(nfr - fr0 < kFR ? nfr - fr0 : kFR);
  for (int k = threadIdx.x; k < bins; k += blockDim.x) {
    const int64_t gi = ((int64_t)c * bins + k) * T + t0;
#pragma unroll
    for (int f = 0; f < kFR; ++f) {
      float2 ya = make_float2(0.f, 0.f), yb = make_float2(0.f, 0.f);
      if (f < nf) {
        const float2 x = __ldg(spec + gi + f);
        if (mask != nullptr) {
          const float m = __ldg(mask + gi + f);
          ya = make_float2(m * x.x, m * x.y);
          const float q = 1.f - m;
          yb = make_float2(q * x.x, q * x.y);
        } else {
          ya = x;
        }
      }
      if (k == 0 || k == NF / 2) {   // c2r transforms ignore the imaginary part of DC and Nyquist
        ya.y = 0.f;
        yb.y = 0.f;
      }
      // z[k] = ya + i yb and z[NF - k] = conj(ya) + i conj(yb), both stored conjugated
      float2* zf = z + f * kFrameSlots;
      zf[fpad(k)] = make_float2(ya.x - yb.y, -(ya.y + yb.x));
      if (k != 0 && k != NF / 2) zf[fpad(NF - k)] = make_float2(ya.x + yb.y, ya.y - yb.x);
    }
  }
  __syncthreads();
  fft2048_frames(z, tw);
  const float inv = 1.f / (float)NF;
  for (int f = 0; f < nf; ++f) {
    const float2* zf = z + f * kFrameSlots;
    float* fa = frames_a + ((int64_t)c * nfr + fr0 + f) * NF;
    float* fb = frames_b ? frames_b + ((int64_t)c * nfr + fr0 + f) * NF : nullptr;
    for (int n = threadIdx.x; n < NF; n += blockDim.x) {
      const float w = win[n] * inv;
      const float2 v = zf[fpad(n)];
      fa[n] = v.x * w;
      if (fb) fb[n] = -v.y * w;
    }
  }
}

// grid (ceil(nfr / kFR), 2 channels)
__global__ void __launch_bounds__(256) istft2048_frames_kernel(const float2* __restrict__ spec,
                                                               const float* __restrict__ mask, int64_t T, int64_t t_first,
                                                               int64_t nfr, float* __restrict__ frames_a,
                                                               float* __restrict__ frames_b,
                                                               const float2* __restrict__ tw,
                                                               const float* __restrict__ win) {
  extern __shared__ float2 z[];
  istft2048_frames(spec, mask, T, t_first, nfr, (int64_t)blockIdx.x * kFR, blockIdx.y, frames_a, frames_b, tw, win, z);
}

// ---- several tracks per launch: grid (total CTAs, 2 channels for the inverse) ----
__global__ void __launch_bounds__(256) stft2048_many_kernel(const FftTrack* __restrict__ tracks, int n_tracks, int hop,
                                                            const float2* __restrict__ tw,
                                                            const float* __restrict__ win) {
  extern __shared__ float2 z[];
  const int i = find_track<&FftTrack::cta0>(tracks, n_tracks, blockIdx.x);
  const FftTrack& tr = tracks[i];
  stft2048_frames(tr.wave, tr.L, hop, tr.spec, tr.T, ((int64_t)blockIdx.x - tr.cta0) * kFR, tr.T, tw, win, z);
}

__global__ void __launch_bounds__(256) istft2048_frames_many_kernel(const FftTrack* __restrict__ tracks, int n_tracks,
                                                                    float* __restrict__ frames_a,
                                                                    float* __restrict__ frames_b,
                                                                    const float2* __restrict__ tw,
                                                                    const float* __restrict__ win) {
  extern __shared__ float2 z[];
  const int i = find_track<&FftTrack::cta0>(tracks, n_tracks, blockIdx.x);
  const FftTrack& tr = tracks[i];
  const int64_t off = 2 * tr.frame_off * kF2048;
  istft2048_frames(tr.spec, tr.mask, tr.T, 0, tr.T, ((int64_t)blockIdx.x - tr.cta0) * kFR, blockIdx.y, frames_a + off,
                   frames_b ? frames_b + off : nullptr, tw, win, z);
}

static constexpr size_t kSmem2048 = (size_t)kFR * kFrameSlots * sizeof(float2);   // 73,728 bytes

static bool fft2048_ready() {   // per-device opt-in to more than 48 KB of dynamic shared memory
  static bool done[64] = {};
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return false;
  if (!done[dev]) {
    if (cudaFuncSetAttribute(stft2048_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmem2048) != cudaSuccess ||
        cudaFuncSetAttribute(istft2048_frames_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmem2048) !=
            cudaSuccess ||
        cudaFuncSetAttribute(stft2048_many_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmem2048) !=
            cudaSuccess ||
        cudaFuncSetAttribute(istft2048_frames_many_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)kSmem2048) != cudaSuccess)
      return false;
    done[dev] = true;
  }
  return true;
}

cudaError_t launch_stft(const float* wave, int64_t L, int n_fft, int hop, float2* spec, int64_t T, int64_t t0,
                        int64_t t1, const float2* twiddle, const float* window, cudaStream_t stream) {
  if (t1 <= t0) return cudaSuccess;
  int logn = 0;
  while ((1 << logn) < n_fft) ++logn;
  if ((1 << logn) != n_fft || n_fft > 4096 || n_fft < 64) return cudaErrorInvalidValue;
  if (n_fft == kF2048 && fft2048_ready()) {
    stft2048_kernel<<<(unsigned)((t1 - t0 + kFR - 1) / kFR), 256, kSmem2048, stream>>>(wave, L, hop, spec, T, t0, t1, twiddle,
                                                                                      window);
    return cudaGetLastError();
  }
  stft_kernel<<<(unsigned)(t1 - t0), 256, n_fft * sizeof(float2), stream>>>(wave, L, n_fft, logn, hop, spec, T, t0,
                                                                             twiddle, window);
  return cudaGetLastError();
}

// Windowed inverse transform of frame t of channel c -> fa (and fb) [NF], one CTA, z: NF float2 of shared memory
__device__ __forceinline__ void istft_frame(const float2* __restrict__ spec, const float* __restrict__ mask, int NF,
                                            int logn, int64_t T, int64_t t, int c, float* __restrict__ fa,
                                            float* __restrict__ fb, const float2* __restrict__ tw,
                                            const float* __restrict__ win, float2* z) {
  const int bins = NF / 2 + 1;
  for (int k = threadIdx.x; k < bins; k += blockDim.x) {
    const int64_t gi = ((int64_t)c * bins + k) * T + t;
    float2 x = spec[gi];
    float2 ya, yb;
    if (mask != nullptr) {
      const float m = mask[gi];
      ya = make_float2(m * x.x, m * x.y);
      const float q = 1.f - m;
      yb = make_float2(q * x.x, q * x.y);
    } else {
      ya = x;
      yb = make_float2(0.f, 0.f);
    }
    if (k == 0 || k == NF / 2) {  // c2r transforms ignore the imaginary part of DC and Nyquist
      ya.y = 0.f;
      yb.y = 0.f;
    }
    const unsigned r0 = __brev((unsigned)k) >> (32 - logn);
    z[r0] = make_float2(ya.x - yb.y, ya.y + yb.x);
    if (k != 0 && k != NF / 2) {
      const unsigned r1 = __brev((unsigned)(NF - k)) >> (32 - logn);
      z[r1] = make_float2(ya.x + yb.y, -ya.y + yb.x);
    }
  }
  __syncthreads();
  fft_inplace<true>(z, tw, NF, logn);
  const float inv = 1.f / (float)NF;
  for (int n = threadIdx.x; n < NF; n += blockDim.x) {
    const float w = win[n] * inv;
    fa[n] = z[n].x * w;
    if (fb) fb[n] = z[n].y * w;
  }
}

// grid (T, 2 channels): windowed inverse transform of one frame of one channel -> frames[stem][c][t][NF]
__global__ void __launch_bounds__(256) istft_frames_kernel(const float2* __restrict__ spec,
                                                           const float* __restrict__ mask, int NF, int logn,
                                                           int64_t T, int64_t t_first, int64_t nfr,
                                                           float* __restrict__ frames_a,
                                                           float* __restrict__ frames_b,
                                                           const float2* __restrict__ tw,
                                                           const float* __restrict__ win) {
  extern __shared__ float2 z[];
  const int c = blockIdx.y;
  float* fa = frames_a + ((int64_t)c * nfr + blockIdx.x) * NF;
  float* fb = frames_b ? frames_b + ((int64_t)c * nfr + blockIdx.x) * NF : nullptr;
  istft_frame(spec, mask, NF, logn, T, t_first + blockIdx.x, c, fa, fb, tw, win, z);
}

// Output sample s of channel c; the scratch holds frames [t_first, t_first + nfr) of the track.
__device__ __forceinline__ void istft_ola_sample(const float* __restrict__ frames_a, const float* __restrict__ frames_b,
                                                 int NF, int hop, int64_t T, int64_t t_first, int64_t nfr, int64_t Lo,
                                                 int c, int64_t s, float* __restrict__ wave_a,
                                                 float* __restrict__ wave_b, const float* __restrict__ win) {
  const int64_t u = s + NF / 2;
  int64_t t1 = u / hop;
  if (t1 > T - 1) t1 = T - 1;
  int64_t t0 = (u - NF + hop) / hop;   // ceil((u - NF + 1) / hop) for u - NF + 1 > 0
  if (u - NF + 1 <= 0) t0 = 0;
  float acc_a = 0.f, acc_b = 0.f, wss = 0.f;
  for (int64_t t = t0; t <= t1; ++t) {
    const int n = (int)(u - t * hop);
    const float w = win[n];
    wss += w * w;
    const int64_t fi = ((int64_t)c * nfr + (t - t_first)) * NF + n;
    acc_a += frames_a[fi];
    if (frames_b) acc_b += frames_b[fi];
  }
  if (wss > 1.17549435e-38f) {   // np.finfo(float32).tiny
    acc_a /= wss;
    acc_b /= wss;
  }
  wave_a[(int64_t)c * Lo + s] = acc_a;
  if (wave_b) wave_b[(int64_t)c * Lo + s] = acc_b;
}

// Output samples [s0, s1) of each channel; the scratch holds frames [t_first, t_first + nfr) of the track.
__global__ void istft_ola_kernel(const float* __restrict__ frames_a, const float* __restrict__ frames_b, int NF,
                                 int hop, int64_t T, int64_t t_first, int64_t nfr, int64_t s0, int64_t s1, int64_t Lo,
                                 float* __restrict__ wave_a, float* __restrict__ wave_b,
                                 const float* __restrict__ win) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t span = s1 - s0;
  if (idx >= 2 * span) return;
  istft_ola_sample(frames_a, frames_b, NF, hop, T, t_first, nfr, Lo, (int)(idx / span), s0 + idx % span, wave_a, wave_b,
                   win);
}

// ---- several tracks per launch (radix-2 frames for n_fft != 2048, overlap-add for every n_fft) ----
__global__ void __launch_bounds__(256) stft_many_kernel(const FftTrack* __restrict__ tracks, int n_tracks, int NF,
                                                        int logn, int hop, const float2* __restrict__ tw,
                                                        const float* __restrict__ win) {
  extern __shared__ float2 z[];
  const FftTrack& tr = tracks[find_track<&FftTrack::cta0>(tracks, n_tracks, blockIdx.x)];
  stft_frame(tr.wave, tr.L, NF, logn, hop, tr.spec, tr.T, (int64_t)blockIdx.x - tr.cta0, tw, win, z);
}

__global__ void __launch_bounds__(256) istft_frames_many_kernel(const FftTrack* __restrict__ tracks, int n_tracks,
                                                                int NF, int logn, float* __restrict__ frames_a,
                                                                float* __restrict__ frames_b,
                                                                const float2* __restrict__ tw,
                                                                const float* __restrict__ win) {
  extern __shared__ float2 z[];
  const FftTrack& tr = tracks[find_track<&FftTrack::cta0>(tracks, n_tracks, blockIdx.x)];
  const int c = blockIdx.y;
  const int64_t t = (int64_t)blockIdx.x - tr.cta0;
  const int64_t fi = (2 * tr.frame_off + (int64_t)c * tr.T + t) * NF;
  istft_frame(tr.spec, tr.mask, NF, logn, tr.T, t, c, frames_a + fi, frames_b ? frames_b + fi : nullptr, tw, win, z);
}

__global__ void istft_ola_many_kernel(const FftTrack* __restrict__ tracks, int n_tracks, int64_t total, int NF, int hop,
                                      const float* __restrict__ frames_a, const float* __restrict__ frames_b,
                                      const float* __restrict__ win) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const FftTrack& tr = tracks[find_track<&FftTrack::s0>(tracks, n_tracks, idx)];
  const int64_t Lo = (int64_t)hop * (tr.T - 1), local = idx - tr.s0;
  const int64_t off = 2 * tr.frame_off * NF;
  istft_ola_sample(frames_a + off, frames_b ? frames_b + off : nullptr, NF, hop, tr.T, 0, tr.T, Lo, (int)(local / Lo),
                   local % Lo, tr.wave_a, tr.wave_b, win);
}

// frames scratch is provided by the caller through wave-independent workspace (see engine.cu)
cudaError_t launch_istft_frames(const float2* spec, const float* mask, int n_fft, int64_t T, int64_t t_first,
                                int64_t nfr, float* frames_a, float* frames_b, const float2* twiddle,
                                const float* window, cudaStream_t stream) {
  if (nfr <= 0) return cudaSuccess;
  int logn = 0;
  while ((1 << logn) < n_fft) ++logn;
  if ((1 << logn) != n_fft || n_fft > 4096 || n_fft < 64) return cudaErrorInvalidValue;
  if (n_fft == kF2048 && fft2048_ready()) {
    dim3 grid4((unsigned)((nfr + kFR - 1) / kFR), 2);
    istft2048_frames_kernel<<<grid4, 256, kSmem2048, stream>>>(spec, mask, T, t_first, nfr, frames_a, frames_b, twiddle,
                                                              window);
    return cudaGetLastError();
  }
  dim3 grid((unsigned)nfr, 2);
  istft_frames_kernel<<<grid, 256, n_fft * sizeof(float2), stream>>>(spec, mask, n_fft, logn, T, t_first, nfr, frames_a,
                                                                     frames_b, twiddle, window);
  return cudaGetLastError();
}

cudaError_t launch_istft_ola(const float* frames_a, const float* frames_b, int n_fft, int hop, int64_t T,
                             int64_t t_first, int64_t nfr, int64_t s0, int64_t s1, float* wave_a, float* wave_b,
                             const float* window, cudaStream_t stream) {
  const int64_t Lo = (int64_t)hop * (T - 1);
  if (s1 <= s0) return cudaSuccess;
  istft_ola_kernel<<<(unsigned)((2 * (s1 - s0) + 255) / 256), 256, 0, stream>>>(frames_a, frames_b, n_fft, hop, T, t_first,
                                                                                nfr, s0, s1, Lo, wave_a, wave_b, window);
  return cudaGetLastError();
}

// The n_fft = 2048 kernels take kFR frames per CTA, the radix-2 kernels one.
int64_t fft_ctas_per_track(int n_fft, int64_t T) { return n_fft == kF2048 ? (T + kFR - 1) / kFR : T; }

static bool fft_logn(int n_fft, int& logn) {
  logn = 0;
  while ((1 << logn) < n_fft) ++logn;
  return (1 << logn) == n_fft && n_fft <= 4096 && n_fft >= 64;
}

cudaError_t launch_stft_many(const FftTrack* tracks, int n_tracks, int64_t total_ctas, int n_fft, int hop,
                             const float2* twiddle, const float* window, cudaStream_t stream) {
  int logn;
  if (!fft_logn(n_fft, logn)) return cudaErrorInvalidValue;
  if (total_ctas <= 0) return cudaSuccess;
  if (n_fft == kF2048) {
    if (!fft2048_ready()) return cudaErrorInvalidValue;
    stft2048_many_kernel<<<(unsigned)total_ctas, 256, kSmem2048, stream>>>(tracks, n_tracks, hop, twiddle, window);
  } else {
    stft_many_kernel<<<(unsigned)total_ctas, 256, n_fft * sizeof(float2), stream>>>(tracks, n_tracks, n_fft, logn, hop,
                                                                                    twiddle, window);
  }
  return cudaGetLastError();
}

cudaError_t launch_istft_frames_many(const FftTrack* tracks, int n_tracks, int64_t total_ctas, int n_fft, float* frames_a,
                                     float* frames_b, const float2* twiddle, const float* window, cudaStream_t stream) {
  int logn;
  if (!fft_logn(n_fft, logn)) return cudaErrorInvalidValue;
  if (total_ctas <= 0) return cudaSuccess;
  dim3 grid((unsigned)total_ctas, 2);
  if (n_fft == kF2048) {
    if (!fft2048_ready()) return cudaErrorInvalidValue;
    istft2048_frames_many_kernel<<<grid, 256, kSmem2048, stream>>>(tracks, n_tracks, frames_a, frames_b, twiddle, window);
  } else {
    istft_frames_many_kernel<<<grid, 256, n_fft * sizeof(float2), stream>>>(tracks, n_tracks, n_fft, logn, frames_a,
                                                                            frames_b, twiddle, window);
  }
  return cudaGetLastError();
}

cudaError_t launch_istft_ola_many(const FftTrack* tracks, int n_tracks, int64_t total_samples, int n_fft, int hop,
                                  const float* frames_a, const float* frames_b, const float* window, cudaStream_t stream) {
  if (total_samples <= 0) return cudaSuccess;
  istft_ola_many_kernel<<<(unsigned)((total_samples + 255) / 256), 256, 0, stream>>>(tracks, n_tracks, total_samples,
                                                                                    n_fft, hop, frames_a, frames_b,
                                                                                    window);
  return cudaGetLastError();
}

}  // namespace vr
