// Mel-spectrogram conditioner (model/condition.py:7-19): ReflectionPad1d((n_fft/2 - hop/2, n_fft/2 + hop/2)) ->
// windowed STFT (center=False) -> |.|^power -> mel filterbank -> log(. + eps), fused in ONE kernel that writes the
// (B, n_mels, frames) tensor the conditioning upsampler (upsample.cu) consumes.  Nothing but the audio is read from
// HBM and nothing but the log-mel frames is written: the padded signal, the (B, n_fft/2+1, frames) complex STFT and the
// power spectrogram of the reference's torchaudio pipeline never exist.
//
// One CTA per (batch, frame).  The n_fft real samples are packed as n_fft/2 complex numbers z[n] = x[2n] + i x[2n+1]
// (window applied, reflected indices resolved while loading), transformed by an in-shared-memory radix-2 FFT of half
// the length, and split back into the n_fft/2+1 one-sided bins (fft.cuh, shared with the denoiser).  A thread per mel
// band then runs over that band's support [lo, hi) of the triangular filter.  The real workloads are small (24 x 63 training frames, 863 frames per
// 10 s utterance), so the kernel is latency bound and a CTA per frame -- the widest decomposition -- is the fast one.
#include "fft.cuh"

namespace cmwg {

template <int NFFT>
__global__ void __launch_bounds__(256) melspec_kernel(const float* __restrict__ x, long long x_bstride, int T,
                                                      const float* __restrict__ window,
                                                      const float* __restrict__ fbt, const int* __restrict__ fb_lo,
                                                      const int* __restrict__ fb_hi, int n_mels, int hop,
                                                      int pad_left, int frames, int power_is_one, float eps,
                                                      int take_log, float* __restrict__ out) {
  constexpr int M = FftShape<NFFT>::M;
  constexpr int NT = 256;
  __shared__ float2 z[FftShape<NFFT>::MP];
  __shared__ float2 tw[FftShape<NFFT>::MP];   // tw[padi(k)] = exp(-2 pi i k / NFFT), k < NFFT/2
  __shared__ float pw[M + 1];                  // |X[k]|^power, k <= NFFT/2

  const int b = blockIdx.x / frames, fr = blockIdx.x % frames;
  const float* xb = x + (long long)b * x_bstride;
  const int start = fr * hop - pad_left;
  int my_lo = 0, my_hi = 0;
  if (threadIdx.x < n_mels) {
    my_lo = fb_lo[threadIdx.x];
    my_hi = fb_hi[threadIdx.x];
  }

  fft_twiddles<NFFT, NT>(tw);
  // bit-reversed scatter of the packed, windowed frame
  for (int n = threadIdx.x; n < M; n += NT) {
    int i0 = reflect_index(start + 2 * n, T), i1 = reflect_index(start + 2 * n + 1, T);
    float a = xb[i0] * window[2 * n], c = xb[i1] * window[2 * n + 1];
    z[fft_bitrev_slot<NFFT>(n)] = make_float2(a, c);
  }
  __syncthreads();
  fft_radix2<NFFT, NT>(z, tw);
  for (int k = threadIdx.x; k <= M; k += NT) {
    float2 X = rfft_split(z[fft_padi(k & (M - 1))], z[fft_padi((M - k) & (M - 1))], fft_split_twiddle<NFFT>(tw, k));
    float p = fmaf(X.x, X.x, X.y * X.y);
    pw[k] = power_is_one ? sqrtf(p) : p;
  }
  __syncthreads();
  // a thread per mel band: its [lo, hi) bounds were fetched before the FFT, and the loop's loads are independent of
  // each other, so the band sums cost one L2 round trip instead of one per band
  for (int m = threadIdx.x, i = 0; m < n_mels; m += NT, ++i) {
    int lo = i == 0 ? my_lo : fb_lo[m], hi = i == 0 ? my_hi : fb_hi[m];
    const float* frow = fbt + (long long)m * (M + 1);
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int f = lo;
    for (; f + 4 <= hi; f += 4) {
      a0 = fmaf(pw[f], frow[f], a0);
      a1 = fmaf(pw[f + 1], frow[f + 1], a1);
      a2 = fmaf(pw[f + 2], frow[f + 2], a2);
      a3 = fmaf(pw[f + 3], frow[f + 3], a3);
    }
    for (; f < hi; ++f) a0 = fmaf(pw[f], frow[f], a0);
    float v = (a0 + a1) + (a2 + a3) + eps;
    out[((long long)b * n_mels + m) * frames + fr] = take_log ? logf(v) : v;
  }
}

}  // namespace cmwg

using namespace cmwg;

extern "C" int cmwg_melspec_frames(int T, int n_fft, int hop) {
  // reflect pad adds n_fft samples in total; center=False framing
  if (T <= 0 || hop <= 0) return 0;
  return T / hop + 1;
}

extern "C" int cmwg_melspec_fwd(const float* x, long long x_bstride, int B, int T, const float* window,
                                const float* fbt, const int* fb_lo, const int* fb_hi, int n_fft, int hop, int n_mels,
                                int power_is_one, float eps, int take_log, float* out, void* stream) {
  CMWG_REQUIRE(B >= 0 && T >= 0 && n_mels > 0 && hop > 0, "melspec: bad sizes B=%d T=%d n_mels=%d hop=%d", B, T,
               n_mels, hop);
  if (B == 0 || T == 0) return CMWG_OK;
  const int pad_left = n_fft / 2 - hop / 2, pad_right = n_fft / 2 + hop / 2;
  CMWG_REQUIRE(pad_right < T, "melspec: reflection padding (%d, %d) needs more than %d samples, got T=%d", pad_left,
               pad_right, pad_right, T);
  const int frames = (T + pad_left + pad_right - n_fft) / hop + 1;
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid((unsigned)(B * frames)), block(256);
#define CMWG_MEL_CASE(N)                                                                                        \
  case N:                                                                                                       \
    melspec_kernel<N><<<grid, block, 0, st>>>(x, x_bstride, T, window, fbt, fb_lo, fb_hi, n_mels, hop, pad_left, \
                                              frames, power_is_one, eps, take_log, out);                       \
    break;
  switch (n_fft) {
    CMWG_MEL_CASE(128)
    CMWG_MEL_CASE(256)
    CMWG_MEL_CASE(512)
    CMWG_MEL_CASE(1024)
    CMWG_MEL_CASE(2048)
    CMWG_MEL_CASE(4096)
    default:
      set_error("melspec: n_fft must be a power of two in [128, 4096], got %d", n_fft);
      return CMWG_ERR_UNSUPPORTED;
  }
#undef CMWG_MEL_CASE
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}
