// Bandwidth-bound kernels of the CascadedNet forward and the Separator glue (HBM roofline).
//   pack_mag_*      inference.py:44-50,58-60 (window gather + |X|) and inference.py:74 (normalise)
//   upsample2x      lib/layers.py:52  F.interpolate(x2, bilinear, align_corners=True), written into the concat slice
//   pool_freq_mean  lib/layers.py:71  AdaptiveAvgPool2d((1, None))
//   broadcast_rows  lib/layers.py:94  bilinear resize from height 1 == exact broadcast
//   mask_out        lib/nets.py:79,109-115,127-129  1x1 conv -> sigmoid -> replicate Nyquist row -> crop offset
//   absmax / lexmax inference.py:74 / inference.py:87,94 global normalisers
//   apply_mask      inference.py:32-36
#include "common.cuh"
#include "kernels.h"

namespace vr {

// ------------------------------------------------------------------------------------------------
// Frame tw of window `window` (|X|/norm, spectrogram padded by pad_l zeros) -> pixel (n, bin, tw) of dst.
__device__ __forceinline__ void pack_mag_pixel(const float2* __restrict__ spec, int bins, int64_t T, int roi, int pad_l,
                                               int window, float nv, ActView dst, int n, int bin, int tw) {
  int64_t t = (int64_t)window * roi + tw - pad_l;
  // A silent track has max|X| = 0 (the reference then divides 0/0 and writes NaN stems for that one file).  Here a
  // NaN would outlive the call: stage-1/2 layers read the aux channel slots of the shared input buffer through zero
  // weights, and 0 * NaN = NaN inside the MMA would poison every later track on this context.  So a zero / non-finite
  // normaliser packs zeros, and non-finite magnitudes (NaN / Inf samples) are packed as zeros as well.
  const float inv = (nv > 0.f && nv <= 3.0e38f) ? 1.0f / nv : 0.f;
  float m0 = 0.f, m1 = 0.f;
  if (t >= 0 && t < T) {
    float2 a = spec[((int64_t)0 * bins + bin) * T + t];
    float2 b = spec[((int64_t)1 * bins + bin) * T + t];
    m0 = hypotf(a.x, a.y) * inv;
    m1 = hypotf(b.x, b.y) * inv;
    if (!(m0 <= 3.0e38f)) m0 = 0.f;   // also catches NaN
    if (!(m1 <= 3.0e38f)) m1 = 0.f;
  }
  int64_t off = (int64_t)n * dst.sn + (int64_t)bin * dst.sh + (int64_t)tw * dst.sw;
  bf16 h0, l0, h1, l1;
  split_bf16(m0, h0, l0);
  split_bf16(m1, h1, l1);
  *reinterpret_cast<__nv_bfloat162*>(dst.hi + off) = __halves2bfloat162(h0, h1);
  *reinterpret_cast<__nv_bfloat162*>(dst.lo + off) = __halves2bfloat162(l0, l1);
}

__global__ void pack_mag_from_spec_kernel(const float2* __restrict__ spec, int bins, int64_t T, int max_bin, int W,
                                          int roi, int pad_l, int first_window, const float* __restrict__ norm,
                                          ActView dst) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = (int64_t)dst.N * max_bin * W;
  if (idx >= total) return;
  int tw = (int)(idx % W);
  int64_t r = idx / W;
  int bin = (int)(r % max_bin);
  int n = (int)(r / max_bin);
  pack_mag_pixel(spec, bins, T, roi, pad_l, first_window + n, *norm, dst, n, bin, tw);
}

// Batch slot n packs window wins[n] of its own track with its track's normaliser.
__global__ void pack_mag_many_kernel(const WinDesc* __restrict__ wins, int bins, int max_bin, int W, int roi,
                                     const float* __restrict__ norms, ActView dst) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = (int64_t)dst.N * max_bin * W;
  if (idx >= total) return;
  int tw = (int)(idx % W);
  int64_t r = idx / W;
  int bin = (int)(r % max_bin);
  int n = (int)(r / max_bin);
  const WinDesc& d = wins[n];
  pack_mag_pixel(d.spec, bins, d.T, roi, d.pad_l, d.window, norms[d.norm], dst, n, bin, tw);
}

cudaError_t launch_pack_mag_many(const WinDesc* wins, int bins, int max_bin, int W, int roi, const float* norms,
                                 ActView dst, cudaStream_t stream) {
  int64_t total = (int64_t)dst.N * max_bin * W;
  if (total == 0) return cudaSuccess;
  pack_mag_many_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(wins, bins, max_bin, W, roi, norms, dst);
  return cudaGetLastError();
}

cudaError_t launch_pack_mag_from_spec(const float2* spec, int bins, int64_t T, int max_bin, int W, int roi,
                                      int pad_l, int first_window, const float* norm, ActView dst,
                                      cudaStream_t stream) {
  int64_t total = (int64_t)dst.N * max_bin * W;
  if (total == 0) return cudaSuccess;
  pack_mag_from_spec_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(spec, bins, T, max_bin, W, roi,
                                                                                 pad_l, first_window, norm, dst);
  return cudaGetLastError();
}

__global__ void pack_mag_from_float_kernel(const float* __restrict__ mag, int bins, int max_bin, ActView dst) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int W = dst.W;
  int64_t total = (int64_t)dst.N * max_bin * W;
  if (idx >= total) return;
  int tw = (int)(idx % W);
  int64_t r = idx / W;
  int bin = (int)(r % max_bin);
  int n = (int)(r / max_bin);
  float m0 = mag[(((int64_t)n * 2 + 0) * bins + bin) * W + tw];
  float m1 = mag[(((int64_t)n * 2 + 1) * bins + bin) * W + tw];
  if (!(fabsf(m0) <= 3.0e38f)) m0 = 0.f;   // non-finite inputs must not reach the shared activation buffers (see above)
  if (!(fabsf(m1) <= 3.0e38f)) m1 = 0.f;
  int64_t off = (int64_t)n * dst.sn + (int64_t)bin * dst.sh + (int64_t)tw * dst.sw;
  bf16 h0, l0, h1, l1;
  split_bf16(m0, h0, l0);
  split_bf16(m1, h1, l1);
  *reinterpret_cast<__nv_bfloat162*>(dst.hi + off) = __halves2bfloat162(h0, h1);
  *reinterpret_cast<__nv_bfloat162*>(dst.lo + off) = __halves2bfloat162(l0, l1);
}

cudaError_t launch_pack_mag_from_float(const float* mag, int bins, int max_bin, ActView dst, cudaStream_t stream) {
  int64_t total = (int64_t)dst.N * max_bin * dst.W;
  if (total == 0) return cudaSuccess;
  pack_mag_from_float_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(mag, bins, max_bin, dst);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// One thread per (output pixel, 8-channel chunk); grid.x = (image, output row) - N * H can exceed the 65535 limit of
// grid.y - so all per-thread index math is 32-bit with one division.  Source index and weights follow ATen's upsample_bilinear2d with
// align_corners=True: scale = (in-1)/(out-1) in fp32, src = scale*dst.
template <int CH>   // channels per thread: 8 (one 16-byte access per plane) or 16 (32 bytes: STG.256, twice the loads in flight)
__global__ void __launch_bounds__(256) upsample2x_kernel(ActView in, ActView out, int chunks, float sh, float sw) {
  const int idx = blockIdx.y * blockDim.x + threadIdx.x;
  if (idx >= out.W * chunks) return;
  const int wo = idx / chunks;
  const int ck = idx - wo * chunks;
  const int n = blockIdx.x / out.H;
  const int ho = blockIdx.x - n * out.H;
  const float fy = sh * ho, fx = sw * wo;
  const int y0 = (int)fy, x0 = (int)fx;
  const int y1 = y0 + (y0 < in.H - 1 ? 1 : 0), x1 = x0 + (x0 < in.W - 1 ? 1 : 0);
  const float ly = fy - y0, lx = fx - x0;
  const float hy = 1.f - ly, hx = 1.f - lx;
  const int64_t base = (int64_t)n * in.sn + ck * CH;
  const int64_t r0 = base + (int64_t)y0 * in.sh, r1 = base + (int64_t)y1 * in.sh;
  const int c0 = x0 * in.sw, c1 = x1 * in.sw;
  constexpr int V = CH / 8;
  bf16x8 ah[V], al[V], bh[V], bl[V], ch[V], cl[V], dh[V], dl[V];
#pragma unroll
  for (int v = 0; v < V; ++v) {
    ah[v] = ld128(in.hi + r0 + c0 + 8 * v); al[v] = ld128(in.lo + r0 + c0 + 8 * v);
    bh[v] = ld128(in.hi + r0 + c1 + 8 * v); bl[v] = ld128(in.lo + r0 + c1 + 8 * v);
    ch[v] = ld128(in.hi + r1 + c0 + 8 * v); cl[v] = ld128(in.lo + r1 + c0 + 8 * v);
    dh[v] = ld128(in.hi + r1 + c1 + 8 * v); dl[v] = ld128(in.lo + r1 + c1 + 8 * v);
  }
  const int64_t oo = (int64_t)n * out.sn + (int64_t)ho * out.sh + (int64_t)wo * out.sw + ck * CH;
  bf16x8 h[V], l[V];
#pragma unroll
  for (int v = 0; v < V; ++v) {
    float a[8], b[8], c[8], d[8], y[8];
    unpack8(ah[v], al[v], a);
    unpack8(bh[v], bl[v], b);
    unpack8(ch[v], cl[v], c);
    unpack8(dh[v], dl[v], d);
#pragma unroll
    for (int i = 0; i < 8; ++i) y[i] = hy * (hx * a[i] + lx * b[i]) + ly * (hx * c[i] + lx * d[i]);
    split8(y, h[v], l[v]);
  }
  if (V == 2) {
    st256(out.hi + oo, h[0], h[V - 1]);
    st256(out.lo + oo, l[0], l[V - 1]);
  } else {
    st128(out.hi + oo, h[0]);
    st128(out.lo + oo, l[0]);
  }
}

cudaError_t launch_upsample2x(ActView in, ActView out, cudaStream_t stream) {
  if ((int64_t)out.N * out.H * out.W * (in.C >> 3) == 0) return cudaSuccess;
  const float sh = out.H > 1 ? (float)(in.H - 1) / (float)(out.H - 1) : 0.f;
  const float sw = out.W > 1 ? (float)(in.W - 1) / (float)(out.W - 1) : 0.f;
  const bool wide = in.C % 16 == 0 && out.sw % 16 == 0 && in.sw % 16 == 0 &&
                    ((reinterpret_cast<uintptr_t>(out.hi) | reinterpret_cast<uintptr_t>(out.lo)) & 31) == 0;
  const int chunks = wide ? in.C >> 4 : in.C >> 3;
  dim3 grid((unsigned)(out.N * out.H), (unsigned)ceil_div(out.W * chunks, 256));
  if (wide)
    upsample2x_kernel<16><<<grid, 256, 0, stream>>>(in, out, chunks, sh, sw);
  else
    upsample2x_kernel<8><<<grid, 256, 0, stream>>>(in, out, chunks, sh, sw);
  return cudaGetLastError();
}

// Single-channel variant for the LSTM branch (lib/nets.py:38, layers.py:52): the source is the fp32 plane in[bin][n][t] the dense GEMM wrote
// (strides in_sn, in_sh in floats, t contiguous); the result goes to channel 0 of a G-channel group (G - 1 zeros), G = 16
// inside a concat buffer (32-byte sectors) or 8 for the buffer of its own that the row kernel reads through a second
// tensor map (TMA zero-fills the rest of the chunk).
template <int G>
__global__ void __launch_bounds__(256) upsample2x_c1_kernel(const float* __restrict__ in, int inH, int inW, int64_t in_sn,
                                                            int64_t in_sh, ActView out, float sh, float sw) {
  const int wo = blockIdx.y * blockDim.x + threadIdx.x;   // rows on grid.x: N * H exceeds the 65535 limit of grid.y
  if (wo >= out.W) return;
  const int n = blockIdx.x / out.H;
  const int ho = blockIdx.x - n * out.H;
  const float fy = sh * ho, fx = sw * wo;
  const int y0 = (int)fy, x0 = (int)fx;
  const int y1 = y0 + (y0 < inH - 1 ? 1 : 0), x1 = x0 + (x0 < inW - 1 ? 1 : 0);
  const float ly = fy - y0, lx = fx - x0;
  const float hy = 1.f - ly, hx = 1.f - lx;
  const float* r0 = in + (int64_t)n * in_sn + (int64_t)y0 * in_sh;
  const float* r1 = in + (int64_t)n * in_sn + (int64_t)y1 * in_sh;
  const float a = __ldg(r0 + x0), b = __ldg(r0 + x1), c = __ldg(r1 + x0), d = __ldg(r1 + x1);
  const float y = hy * (hx * a + lx * b) + ly * (hx * c + lx * d);
  bf16 h, l;
  split_bf16(y, h, l);
  const int64_t oo = (int64_t)n * out.sn + (int64_t)ho * out.sh + (int64_t)wo * out.sw;
  const uint4 z = make_uint4(0, 0, 0, 0);
  if (G == 16) {
    st256(out.hi + oo, make_uint4((uint32_t)__bfloat16_as_ushort(h), 0, 0, 0), z);
    st256(out.lo + oo, make_uint4((uint32_t)__bfloat16_as_ushort(l), 0, 0, 0), z);
  } else {
    st128(out.hi + oo, make_uint4((uint32_t)__bfloat16_as_ushort(h), 0, 0, 0));
    st128(out.lo + oo, make_uint4((uint32_t)__bfloat16_as_ushort(l), 0, 0, 0));
  }
}

cudaError_t launch_upsample2x_c1(const float* in, int inH, int inW, int64_t in_sn, int64_t in_sh, ActView out,
                                 cudaStream_t stream) {
  if ((int64_t)out.N * out.H * out.W == 0) return cudaSuccess;
  const uintptr_t align = reinterpret_cast<uintptr_t>(out.hi) | reinterpret_cast<uintptr_t>(out.lo);
  if (!((out.C == 16 && out.sw % 16 == 0 && (align & 31) == 0) || (out.C == 8 && out.sw % 8 == 0 && (align & 15) == 0)))
    return cudaErrorInvalidValue;
  const float sh = out.H > 1 ? (float)(inH - 1) / (float)(out.H - 1) : 0.f;
  const float sw = out.W > 1 ? (float)(inW - 1) / (float)(out.W - 1) : 0.f;
  dim3 grid((unsigned)(out.N * out.H), (unsigned)ceil_div(out.W, 256));
  if (out.C == 16)
    upsample2x_c1_kernel<16><<<grid, 256, 0, stream>>>(in, inH, inW, in_sn, in_sh, out, sh, sw);
  else
    upsample2x_c1_kernel<8><<<grid, 256, 0, stream>>>(in, inH, inW, in_sn, in_sh, out, sh, sw);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
__global__ void pool_freq_mean_kernel(ActView in, ActView out) {
  const int chunks = in.C >> 3;
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = (int64_t)in.N * in.W * chunks;
  if (idx >= total) return;
  int ck = (int)(idx % chunks);
  int64_t r = idx / chunks;
  int w = (int)(r % in.W);
  int n = (int)(r / in.W);
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  for (int h = 0; h < in.H; ++h) {
    float x[8];
    int64_t o = (int64_t)n * in.sn + (int64_t)h * in.sh + (int64_t)w * in.sw + ck * 8;
    load8(in.hi + o, in.lo + o, x);
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] += x[i];
  }
  const float inv = 1.f / (float)in.H;
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] *= inv;
  int64_t oo = (int64_t)n * out.sn + (int64_t)w * out.sw + ck * 8;
  bf16x8 hh, ll;
  split8(acc, hh, ll);
  st128(out.hi + oo, hh);
  st128(out.lo + oo, ll);
}

cudaError_t launch_pool_freq_mean(ActView in, ActView out, cudaStream_t stream) {
  int64_t total = (int64_t)in.N * in.W * (in.C >> 3);
  if (total == 0) return cudaSuccess;
  pool_freq_mean_kernel<<<(unsigned)((total + 127) / 128), 128, 0, stream>>>(in, out);
  return cudaGetLastError();
}

__global__ void broadcast_rows_kernel(ActView in, ActView out) {
  const int chunks = in.C >> 3;
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = (int64_t)out.N * out.H * out.W * chunks;
  if (idx >= total) return;
  int ck = (int)(idx % chunks);
  int64_t r = idx / chunks;
  int w = (int)(r % out.W);
  r /= out.W;
  int h = (int)(r % out.H);
  int n = (int)(r / out.H);
  int64_t oi = (int64_t)n * in.sn + (int64_t)w * in.sw + ck * 8;
  int64_t oo = (int64_t)n * out.sn + (int64_t)h * out.sh + (int64_t)w * out.sw + ck * 8;
  st128(out.hi + oo, ld128(in.hi + oi));
  st128(out.lo + oo, ld128(in.lo + oi));
}

cudaError_t launch_broadcast_rows(ActView in, ActView out, cudaStream_t stream) {
  int64_t total = (int64_t)out.N * out.H * out.W * (in.C >> 3);
  if (total == 0) return cudaSuccess;
  broadcast_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(in, out);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Final 1x1 conv (nout -> 2, no BN) + sigmoid, only for the frames that survive the offset crop.
// Kept frame tr of image n, row bin of f3 -> d0 (channel 0) and d0 + stride_c (channel 1); the Nyquist row is also
// stored one row (stride_bin) further down.
template <int NOUT>
__device__ __forceinline__ void mask_out_pixel(const ActView& f3, const float* __restrict__ w, int offset, int n,
                                               int bin, int tr, float* d0, int64_t stride_c, int64_t stride_bin,
                                               int accumulate) {
  int64_t o = (int64_t)n * f3.sn + (int64_t)bin * f3.sh + (int64_t)(tr + offset) * f3.sw;
  float a0 = 0.f, a1 = 0.f;
#pragma unroll
  for (int c = 0; c < NOUT; c += 8) {
    float x[8];
    load8(f3.hi + o + c, f3.lo + o + c, x);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      a0 = fmaf(x[i], __ldg(w + c + i), a0);
      a1 = fmaf(x[i], __ldg(w + NOUT + c + i), a1);
    }
  }
  float m0 = 1.f / (1.f + expf(-a0));
  float m1 = 1.f / (1.f + expf(-a1));
  float* d1 = d0 + stride_c;
  const bool last = bin == f3.H - 1;   // F.pad(..., mode='replicate') of the Nyquist row (lib/nets.py:111-115)
  if (accumulate) {
    *d0 = (*d0 + m0) * 0.5f;
    *d1 = (*d1 + m1) * 0.5f;
    if (last) {
      d0[stride_bin] = (d0[stride_bin] + m0) * 0.5f;
      d1[stride_bin] = (d1[stride_bin] + m1) * 0.5f;
    }
  } else {
    *d0 = m0;
    *d1 = m1;
    if (last) {
      d0[stride_bin] = m0;
      d1[stride_bin] = m1;
    }
  }
}

template <int NOUT>
__global__ void mask_out_kernel(MaskOutParams p) {
  const int roi = p.f3.W - 2 * p.offset;
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = (int64_t)p.f3.N * p.f3.H * roi;
  if (idx >= total) return;
  int tr = (int)(idx % roi);
  int64_t r = idx / roi;
  int bin = (int)(r % p.f3.H);
  int n = (int)(r / p.f3.H);
  int64_t t = p.t_base0 + (int64_t)n * p.roi_t + tr;
  if (t < 0 || t >= p.t_limit) return;
  float* d0 = p.out + (int64_t)n * p.stride_n + (int64_t)bin * p.stride_bin + p.t_base0 + tr;
  mask_out_pixel<NOUT>(p.f3, p.w, p.offset, n, bin, tr, d0, p.stride_c, p.stride_bin, p.accumulate);
}

// Batch slot n writes into the mask of its own track: wins[n].mask [2][bins][T], frame t_base + tr.
template <int NOUT>
__global__ void mask_out_many_kernel(ActView f3, const float* __restrict__ w, int offset,
                                     const WinDesc* __restrict__ wins) {
  const int roi = f3.W - 2 * offset;
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = (int64_t)f3.N * f3.H * roi;
  if (idx >= total) return;
  int tr = (int)(idx % roi);
  int64_t r = idx / roi;
  int bin = (int)(r % f3.H);
  int n = (int)(r / f3.H);
  const WinDesc& d = wins[n];
  const int64_t t = d.t_base + tr;
  if (t < 0 || t >= d.T) return;
  float* d0 = d.mask + (int64_t)bin * d.T + t;
  mask_out_pixel<NOUT>(f3, w, offset, n, bin, tr, d0, (int64_t)(f3.H + 1) * d.T, d.T, d.accumulate);
}

cudaError_t launch_mask_out_many(ActView f3, const float* w, int offset, const WinDesc* wins, cudaStream_t stream) {
  const int roi = f3.W - 2 * offset;
  int64_t total = (int64_t)f3.N * f3.H * roi;
  if (total <= 0) return cudaSuccess;
  unsigned grid = (unsigned)((total + 255) / 256);
  switch (f3.C) {
    case 8: mask_out_many_kernel<8><<<grid, 256, 0, stream>>>(f3, w, offset, wins); break;
    case 16: mask_out_many_kernel<16><<<grid, 256, 0, stream>>>(f3, w, offset, wins); break;
    case 32: mask_out_many_kernel<32><<<grid, 256, 0, stream>>>(f3, w, offset, wins); break;
    case 64: mask_out_many_kernel<64><<<grid, 256, 0, stream>>>(f3, w, offset, wins); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

cudaError_t launch_mask_out(const MaskOutParams& p, cudaStream_t stream) {
  const int roi = p.f3.W - 2 * p.offset;
  int64_t total = (int64_t)p.f3.N * p.f3.H * roi;
  if (total <= 0) return cudaSuccess;
  unsigned grid = (unsigned)((total + 255) / 256);
  switch (p.f3.C) {
    case 8: mask_out_kernel<8><<<grid, 256, 0, stream>>>(p); break;
    case 16: mask_out_kernel<16><<<grid, 256, 0, stream>>>(p); break;
    case 32: mask_out_kernel<32><<<grid, 256, 0, stream>>>(p); break;
    case 64: mask_out_kernel<64><<<grid, 256, 0, stream>>>(p); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// max|spec[i]| over i = i0, i0 + step, ... < n, reduced over the CTA into *out (atomicMax on the bits: m >= 0).  Every
// thread of the CTA must call it.
__device__ __forceinline__ void absmax_block(const float2* __restrict__ spec, int64_t n, int64_t i0, int64_t step,
                                             float* out) {
  float m = 0.f;
  for (int64_t i = i0; i < n; i += step) {
    float2 v = spec[i];
    m = fmaxf(m, hypotf(v.x, v.y));
  }
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  __shared__ float s[32];
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x < 32) {
    m = threadIdx.x < (blockDim.x >> 5) ? s[threadIdx.x] : 0.f;
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (threadIdx.x == 0) atomicMax(reinterpret_cast<unsigned int*>(out), __float_as_uint(m));  // m >= 0
  }
}

__global__ void absmax_kernel(const float2* __restrict__ spec, int64_t n, float* out) {
  absmax_block(spec, n, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, (int64_t)gridDim.x * blockDim.x, out);
}

cudaError_t launch_absmax(const float2* spec, int64_t n, float* out_absmax, cudaStream_t stream) {
  cudaError_t e = cudaMemsetAsync(out_absmax, 0, sizeof(float), stream);
  if (e != cudaSuccess) return e;
  if (n == 0) return cudaSuccess;
  int grid = (int)(((n + 255) / 256) < 148 * 8 ? ((n + 255) / 256) : 148 * 8);
  absmax_kernel<<<grid, 256, 0, stream>>>(spec, n, out_absmax);
  return cudaGetLastError();
}

__global__ void absmax_range_kernel(const float2* __restrict__ spec, int nrows, int64_t T, int64_t t0, int64_t t1,
                                    float* out) {
  const int64_t span = t1 - t0;
  const int64_t n = (int64_t)nrows * span;
  float m = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / span;
    const float2 v = spec[r * T + t0 + (i - r * span)];
    m = fmaxf(m, hypotf(v.x, v.y));
  }
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<unsigned int*>(out), __float_as_uint(m));   // m >= 0
}

cudaError_t launch_absmax_range(const float2* spec, int nrows, int64_t T, int64_t t0, int64_t t1, float* out_absmax,
                                cudaStream_t stream) {
  cudaError_t e = cudaMemsetAsync(out_absmax, 0, sizeof(float), stream);
  if (e != cudaSuccess) return e;
  const int64_t n = (int64_t)nrows * (t1 - t0);
  if (n <= 0) return cudaSuccess;
  int grid = (int)(((n + 255) / 256) < 148 * 8 ? ((n + 255) / 256) : 148 * 8);
  absmax_range_kernel<<<grid, 256, 0, stream>>>(spec, nrows, T, t0, t1, out_absmax);
  return cudaGetLastError();
}

// numpy's max() of a complex array is lexicographic (largest real part, ties by imaginary part);
// separate_tta divides by that complex number (inference.py:87,94), so the net sees |X| / |lexmax|.
__device__ __forceinline__ unsigned int order_key(float f) {
  unsigned int u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float order_unkey(unsigned int k) {
  unsigned int u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  return __uint_as_float(u);
}

// lexicographic max key of spec[i], i = i0, i0 + step, ... < n, reduced per warp into *scratch
__device__ __forceinline__ void lexmax_block(const float2* __restrict__ spec, int64_t n, int64_t i0, int64_t step,
                                             unsigned long long* scratch) {
  unsigned long long best = 0ull;
  for (int64_t i = i0; i < n; i += step) {
    float2 v = spec[i];
    unsigned long long k = ((unsigned long long)order_key(v.x) << 32) | order_key(v.y);
    best = k > best ? k : best;
  }
  for (int o = 16; o > 0; o >>= 1) {
    unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
    best = other > best ? other : best;
  }
  if ((threadIdx.x & 31) == 0) atomicMax(scratch, best);
}

__device__ __forceinline__ float lexmax_finish(unsigned long long k) {
  float re = order_unkey((unsigned int)(k >> 32));
  float im = order_unkey((unsigned int)(k & 0xffffffffu));
  // the zero padding of X_spec_pad also takes part in the max (inference.py:86-87)
  unsigned long long kz = ((unsigned long long)order_key(0.f) << 32) | order_key(0.f);
  if (kz > k) { re = 0.f; im = 0.f; }
  return hypotf(re, im);
}

__global__ void lexmax_kernel(const float2* __restrict__ spec, int64_t n, unsigned long long* scratch) {
  lexmax_block(spec, n, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, (int64_t)gridDim.x * blockDim.x, scratch);
}

__global__ void lexmax_finish_kernel(const unsigned long long* scratch, float* out_norm) {
  *out_norm = lexmax_finish(*scratch);
}

// grid (n_tracks, CTAs per track): CTA (i, j) reduces elements j*256 + tid, strided by gridDim.y*256, of track i
__global__ void absmax_many_kernel(const NormTrack* __restrict__ tracks, float* out) {
  const NormTrack tr = tracks[blockIdx.x];
  absmax_block(tr.spec, tr.n, (int64_t)blockIdx.y * blockDim.x + threadIdx.x, (int64_t)gridDim.y * blockDim.x,
               out + blockIdx.x);
}

__global__ void lexmax_many_kernel(const NormTrack* __restrict__ tracks, unsigned long long* scratch) {
  const NormTrack tr = tracks[blockIdx.x];
  lexmax_block(tr.spec, tr.n, (int64_t)blockIdx.y * blockDim.x + threadIdx.x, (int64_t)gridDim.y * blockDim.x,
               scratch + blockIdx.x);
}

__global__ void lexmax_finish_many_kernel(const unsigned long long* scratch, int n_tracks, float* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_tracks) out[i] = lexmax_finish(scratch[i]);
}

cudaError_t launch_normaliser_many(const NormTrack* tracks, int n_tracks, int64_t max_n, int mode,
                                   unsigned long long* scratch, float* out, cudaStream_t stream) {
  if (n_tracks <= 0) return cudaSuccess;
  cudaError_t e = mode == 0 ? cudaMemsetAsync(out, 0, sizeof(float) * n_tracks, stream)
                            : cudaMemsetAsync(scratch, 0, sizeof(unsigned long long) * n_tracks, stream);
  if (e != cudaSuccess) return e;
  // about as many CTAs in all as the single-track kernels use for one track (148 SMs x 8), at least one per track
  int64_t per = (max_n + 255) / 256;
  const int64_t cap = (148 * 8 + n_tracks - 1) / n_tracks;
  if (per > cap) per = cap;
  if (per > 65535) per = 65535;
  if (per < 1) per = 1;
  dim3 grid((unsigned)n_tracks, (unsigned)per);
  if (mode == 0) {
    absmax_many_kernel<<<grid, 256, 0, stream>>>(tracks, out);
  } else {
    lexmax_many_kernel<<<grid, 256, 0, stream>>>(tracks, scratch);
    lexmax_finish_many_kernel<<<(unsigned)((n_tracks + 127) / 128), 128, 0, stream>>>(scratch, n_tracks, out);
  }
  return cudaGetLastError();
}

cudaError_t launch_lexmax_abs(const float2* spec, int64_t n, unsigned long long* scratch, float* out_norm,
                              cudaStream_t stream) {
  cudaError_t e = cudaMemsetAsync(scratch, 0, sizeof(unsigned long long), stream);
  if (e != cudaSuccess) return e;
  if (n > 0) {
    int grid = (int)(((n + 255) / 256) < 148 * 8 ? ((n + 255) / 256) : 148 * 8);
    lexmax_kernel<<<grid, 256, 0, stream>>>(spec, n, scratch);
  }
  lexmax_finish_kernel<<<1, 1, 0, stream>>>(scratch, out_norm);
  return cudaGetLastError();
}

// --postprocess (reference lib/spec_utils.py:60-93, inference.py:27-30) on the device: the per-frame minimum of the
// mask over (channel, bin) goes to the host (4 B per frame), which finds the long above-threshold runs exactly as the
// reference does and returns one fade weight per frame; the mask is then pulled towards 1 by that weight.
__global__ void mask_frame_min_kernel(const float* __restrict__ mask, int rows, int64_t T, float* __restrict__ out) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  float m = mask[t];
  for (int r = 1; r < rows; ++r) m = fminf(m, mask[(int64_t)r * T + t]);
  out[t] = m;
}

cudaError_t launch_mask_frame_min(const float* mask, int rows, int64_t T, float* out, cudaStream_t stream) {
  if (T == 0) return cudaSuccess;
  mask_frame_min_kernel<<<(unsigned)((T + 127) / 128), 128, 0, stream>>>(mask, rows, T, out);
  return cudaGetLastError();
}

__global__ void mask_apply_weight_kernel(float* __restrict__ mask, int64_t n, int64_t T,
                                         const float* __restrict__ weight) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float m = mask[i];
  mask[i] = m + weight[i % T] * (1.f - m);
}

cudaError_t launch_mask_apply_weight(float* mask, int rows, int64_t T, const float* weight, cudaStream_t stream) {
  const int64_t n = (int64_t)rows * T;
  if (n == 0) return cudaSuccess;
  mask_apply_weight_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(mask, n, T, weight);
  return cudaGetLastError();
}

__global__ void apply_mask_kernel(const float2* __restrict__ spec, const float* __restrict__ mask, int64_t n,
                                  float2* __restrict__ y, float2* __restrict__ v) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float2 x = spec[i];
  float m = mask[i];
  y[i] = make_float2(m * x.x, m * x.y);
  float q = 1.f - m;
  v[i] = make_float2(q * x.x, q * x.y);
}

cudaError_t launch_apply_mask(const float2* spec, const float* mask, int64_t n, float2* y, float2* v,
                              cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  apply_mask_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(spec, mask, n, y, v);
  return cudaGetLastError();
}

}  // namespace vr

// ------------------------------------------------------------------------------------------------
// Layout converters used by the API-parity entry points and the tests (NCHW fp32 <-> NHWC split-bf16).
namespace vr {

__global__ void nchw_to_act_kernel(const float* __restrict__ x, int C, ActView dst) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = (int64_t)dst.N * dst.H * dst.W * dst.C;
  if (idx >= total) return;
  int c = (int)(idx % dst.C);
  int64_t r = idx / dst.C;
  int w = (int)(r % dst.W);
  r /= dst.W;
  int h = (int)(r % dst.H);
  int n = (int)(r / dst.H);
  float v = c < C ? x[(((int64_t)n * C + c) * dst.H + h) * dst.W + w] : 0.f;
  int64_t o = (int64_t)n * dst.sn + (int64_t)h * dst.sh + (int64_t)w * dst.sw + c;
  split_bf16(v, dst.hi[o], dst.lo[o]);
}

cudaError_t launch_nchw_to_act(const float* x, int C, ActView dst, cudaStream_t stream) {
  int64_t total = (int64_t)dst.N * dst.H * dst.W * dst.C;
  if (total == 0) return cudaSuccess;
  nchw_to_act_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(x, C, dst);
  return cudaGetLastError();
}

__global__ void act_to_nchw_kernel(ActView src, int C, float* __restrict__ y) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = (int64_t)src.N * C * src.H * src.W;
  if (idx >= total) return;
  int w = (int)(idx % src.W);
  int64_t r = idx / src.W;
  int h = (int)(r % src.H);
  r /= src.H;
  int c = (int)(r % C);
  int n = (int)(r / C);
  int64_t o = (int64_t)n * src.sn + (int64_t)h * src.sh + (int64_t)w * src.sw + c;
  y[idx] = join_bf16(src.hi[o], src.lo[o]);
}

cudaError_t launch_act_to_nchw(ActView src, int C, float* y, cudaStream_t stream) {
  int64_t total = (int64_t)src.N * C * src.H * src.W;
  if (total == 0) return cudaSuccess;
  act_to_nchw_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(src, C, y);
  return cudaGetLastError();
}

}  // namespace vr
