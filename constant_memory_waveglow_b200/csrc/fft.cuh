// In-shared-memory real FFT of one frame, shared by the mel-spectrogram conditioner (melspec.cu) and the denoiser
// (denoise.cu).  A real frame of NFFT samples is packed as M = NFFT/2 complex numbers z[n] = x[2n] + i x[2n+1], transformed by
// a radix-2 decimation-in-time FFT of length M, and split into the NFFT/2 + 1 one-sided bins.  The inverse runs the same
// forward FFT on the conjugate of the merged half-length spectrum.  Every CTA-wide step is a loop over `threadIdx.x` with
// stride NT, followed by __syncthreads() where the next step reads what other threads wrote.
#pragma once
#include "common.cuh"

namespace cmwg {

__device__ __forceinline__ int reflect_index(int i, int T) {
  // ReflectionPad1d semantics (edge sample not repeated); valid for pads < T
  if (i < 0) i = -i;
  if (i >= T) i = 2 * (T - 1) - i;
  return i;
}

// one pad slot per 16 entries: the bit-reversed scatter (stride M/2) and the strided twiddle reads of the late stages
// (stride NFFT >> (s+1)) would otherwise hit a single bank 32 ways
__device__ __forceinline__ int fft_padi(int i) { return i + (i >> 4); }

template <int NFFT> struct FftShape {
  static constexpr int M = NFFT / 2;  // complex FFT length
  static constexpr int LOGM = (M == 64) ? 6 : (M == 128) ? 7 : (M == 256) ? 8 : (M == 512) ? 9 : (M == 1024) ? 10 : 11;
  static constexpr int MP = M + M / 16;  // padded shared-memory length of z and tw
  static_assert(M == (1 << LOGM), "NFFT must be a power of two in [128, 4096]");
};

// shared-memory slot of the bit-reversed position of n < M
template <int NFFT> __device__ __forceinline__ int fft_bitrev_slot(int n) {
  return fft_padi((int)(__brev((unsigned)n) >> (32 - FftShape<NFFT>::LOGM)));
}

// tw[padi(k)] = exp(-2 pi i k / NFFT), k < NFFT/2
template <int NFFT, int NT> __device__ __forceinline__ void fft_twiddles(float2* tw) {
  for (int k = threadIdx.x; k < FftShape<NFFT>::M; k += NT) {
    float s, c;
    sincospif(-2.f * (float)k / (float)NFFT, &s, &c);
    tw[fft_padi(k)] = make_float2(c, s);
  }
}

// radix-2 decimation-in-time stages on M points, in place on the bit-reversed z; twiddle exp(-2 pi i pos / (2 half)) =
// tw[pos * (NFFT / (2 half))].  Expects z written and synchronised; ends with __syncthreads().
template <int NFFT, int NT> __device__ __forceinline__ void fft_radix2(float2* z, const float2* tw) {
  constexpr int M = FftShape<NFFT>::M, LOGM = FftShape<NFFT>::LOGM;
#pragma unroll 1
  for (int s = 0; s < LOGM; ++s) {
    const int half = 1 << s;
    const int tstep = NFFT >> (s + 1);
    for (int j = threadIdx.x; j < M / 2; j += NT) {
      int pos = j & (half - 1);
      int i0 = ((j >> s) << (s + 1)) + pos, i1 = i0 + half;
      float2 w = tw[fft_padi(pos * tstep)];
      i0 = fft_padi(i0);
      i1 = fft_padi(i1);
      float2 u = z[i0], v = z[i1];
      float2 t = make_float2(fmaf(v.x, w.x, -v.y * w.y), fmaf(v.x, w.y, v.y * w.x));
      z[i0] = make_float2(u.x + t.x, u.y + t.y);
      z[i1] = make_float2(u.x - t.x, u.y - t.y);
    }
    __syncthreads();
  }
}

// twiddle of bin k <= M for the split / merge: tw[k] for k < M, exp(-i pi) = -1 for k = M
template <int NFFT> __device__ __forceinline__ float2 fft_split_twiddle(const float2* tw, int k) {
  return (k < FftShape<NFFT>::M) ? tw[fft_padi(k)] : make_float2(-1.f, 0.f);
}

// split: X[k] = (Z[k] + conj Z[M-k]) / 2 - (i/2) w (Z[k] - conj Z[M-k]) with a = Z[k], c = Z[M-k] (Z[M] = Z[0]) and
// w = exp(-2 pi i k / NFFT).  The FMAs are spelled out so that every caller rounds alike; they are the contractions the
// compiler chose for the mel-spectrogram kernel before this code was shared, which keeps its output bit for bit.
__device__ __forceinline__ float2 rfft_split(float2 a, float2 c, float2 w) {
  float sr = a.x + c.x, si = a.y - c.y;                     // twice the even part
  float dr = 0.5f * (a.x - c.x), di = 0.5f * (a.y + c.y);   // d = (Z[k] - conj Z[M-k]) / 2
  // p = w * d; X = even part - i p
  float pr = fmaf(dr, w.x, -__fmul_rn(w.y, di)), pi = fmaf(dr, w.y, __fmul_rn(w.x, di));
  return make_float2(fmaf(sr, 0.5f, pi), fmaf(si, 0.5f, -pr));
}

// The inverse of rfft_split: with a = X[k], c = X[M-k] of a one-sided spectrum and w = exp(-2 pi i k / NFFT), k < M, returns
// conj(2 Z[k]), 2 Z[k] = (X[k] + conj X[M-k]) + i conj(w) (X[k] - conj X[M-k]), where Z is the M-point DFT of the packed
// signal x[2n] + i x[2n+1].  If F is the forward FFT (fft_radix2) of these values, F[n] = NFFT conj(x[2n] + i x[2n+1]):
// x[2n] = Re F[n] / NFFT and x[2n+1] = -Im F[n] / NFFT.
__device__ __forceinline__ float2 irfft_merge_conj(float2 a, float2 c, float2 w) {
  float sr = a.x + c.x, si = a.y - c.y;   // X[k] + conj X[M-k]
  float dr = a.x - c.x, di = a.y + c.y;   // X[k] - conj X[M-k]
  // conj(w) * d
  float er = w.x * dr + w.y * di, ei = w.x * di - w.y * dr;
  // s + i (conj(w) d), conjugated
  return make_float2(sr - ei, -(si + er));
}

}  // namespace cmwg
