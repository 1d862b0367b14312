// Spectral distances between (reference, estimate) pairs of a padded batch with per-item lengths: log-spectral distance,
// log-mel L1 and mel-cepstral distortion on Tacotron2's STFT and mel (the framing of melspec_varlen_kernel with
// pad_left = n_fft/2, the mel of TacotronSTFT.mel_spectrogram).
//
// Two kernels.  spectral_distance_frames_kernel: one CTA per (frame, item).  Both windowed frames go through the same
// load / FFT / split code one after the other (fft.cuh), so identical inputs give identical spectra bit for bit; the
// power spectrum, the mel and the log-mel live in shared memory, and the CTA writes its three frame terms -- nothing else
// -- to a (B, 3, T / hop + 1) workspace.  spectral_distance_reduce_kernel: one CTA per item sums the item's len / hop + 1
// terms of each metric in a fixed order and divides.  No atomics and no reads past an item's length or from another
// item, so a batched item equals its solo call bit for bit.
#include "fft.cuh"

namespace cmwg {

constexpr float kMcdScale = 4.342944819032518f;   // 10 / ln 10

// terms[b][0][fr] = sqrt(mean_k (log10 max(P, 1e-10) - log10 max(P^, 1e-10))^2),  P = |S|^2, k <= NFFT/2
// terms[b][1][fr] = mean_j |m_j - m^_j|,  m = ln max(mel_basis @ |S|, 1e-5)
// terms[b][2][fr] = (10 / ln 10) sqrt(2 sum_{d=1}^{n_cep-1} (D (m - m^))_d^2)
// for fr <= len_b / hop; dm (dynamic shared memory) holds n_mels floats.  The minimum of 2 CTAs per SM is a register
// budget: with __launch_bounds__(256) alone ptxas keeps the 512- and 2048-point instances at 32 registers and spills.
template <int NFFT>
__global__ void __launch_bounds__(256, 2) spectral_distance_frames_kernel(
    const float* __restrict__ ref, const float* __restrict__ est, long long bstride, int T,
    const int* __restrict__ lengths, const float* __restrict__ window, const float* __restrict__ fbt,
    const int* __restrict__ fb_lo, const int* __restrict__ fb_hi, const float* __restrict__ dct, int hop, int n_mels,
    int n_cep, int ws_frames, float* __restrict__ terms) {
  constexpr int M = FftShape<NFFT>::M;
  constexpr int NT = 256;
  __shared__ float2 z[FftShape<NFFT>::MP];
  __shared__ float2 tw[FftShape<NFFT>::MP];
  __shared__ float pw[M + 1];                  // |X[k]|^2 of the signal last transformed
  __shared__ float red[3][NT / 32];
  extern __shared__ float dm[];                // log-mel of the reference, then the log-mel difference

  const int fr = blockIdx.x, b = blockIdx.y;
  const int len = lengths != nullptr ? lengths[b] : T;
  if (fr > len / hop) return;
  const int start = fr * hop - NFFT / 2;
  float lsd = 0.f, l1 = 0.f, cep = 0.f;        // this thread's share of the three sums, in a fixed order

  fft_twiddles<NFFT, NT>(tw);
#pragma unroll 1
  for (int s = 0; s < 2; ++s) {
    const float* xb = (s == 0 ? ref : est) + (long long)b * bstride;
    for (int n = threadIdx.x; n < M; n += NT) {
      int i0 = reflect_index(start + 2 * n, len), i1 = reflect_index(start + 2 * n + 1, len);
      z[fft_bitrev_slot<NFFT>(n)] = make_float2(xb[i0] * window[2 * n], xb[i1] * window[2 * n + 1]);
    }
    __syncthreads();
    fft_radix2<NFFT, NT>(z, tw);
    for (int k = threadIdx.x; k <= M; k += NT) {
      float2 X = rfft_split(z[fft_padi(k & (M - 1))], z[fft_padi((M - k) & (M - 1))], fft_split_twiddle<NFFT>(tw, k));
      const float p = fmaf(X.x, X.x, X.y * X.y);
      // the differences are __fsub_rn: a plain `-` lets the compiler fuse the last multiply of one log into an FMA with
      // the subtraction, and identical inputs then give a difference of a rounding error instead of exactly 0
      if (s == 1) {                            // pw[k] still holds the reference's power of bin k
        const float d = __fsub_rn(log10f(fmaxf(pw[k], 1e-10f)), log10f(fmaxf(p, 1e-10f)));
        lsd = fmaf(d, d, lsd);
      }
      pw[k] = p;
    }
    __syncthreads();
    // a thread per mel band over its support [lo, hi), summed as melspec_varlen_kernel sums it
    for (int m = threadIdx.x; m < n_mels; m += NT) {
      const int lo = fb_lo[m], hi = fb_hi[m];
      const float* frow = fbt + (long long)m * (M + 1);
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
      int f = lo;
      for (; f + 4 <= hi; f += 4) {
        a0 = fmaf(sqrtf(pw[f]), frow[f], a0);
        a1 = fmaf(sqrtf(pw[f + 1]), frow[f + 1], a1);
        a2 = fmaf(sqrtf(pw[f + 2]), frow[f + 2], a2);
        a3 = fmaf(sqrtf(pw[f + 3]), frow[f + 3], a3);
      }
      for (; f < hi; ++f) a0 = fmaf(sqrtf(pw[f]), frow[f], a0);
      const float lm = logf(fmaxf((a0 + a1) + (a2 + a3), 1e-5f));
      if (s == 0) {
        dm[m] = lm;
      } else {
        const float d = __fsub_rn(dm[m], lm);
        dm[m] = d;
        l1 += fabsf(d);
      }
    }
    __syncthreads();
  }
  // the DCT is linear: c - c^ = D (m - m^), which also keeps the cepstral difference free of cancellation
  for (int d = 1 + threadIdx.x; d < n_cep; d += NT) {
    const float* row = dct + (long long)d * n_mels;
    float c = 0.f;
    for (int j = 0; j < n_mels; ++j) c = fmaf(row[j], dm[j], c);
    cep = fmaf(c, c, cep);
  }
  lsd = warp_sum(lsd);
  l1 = warp_sum(l1);
  cep = warp_sum(cep);
  if ((threadIdx.x & 31) == 0) {
    red[0][threadIdx.x >> 5] = lsd;
    red[1][threadIdx.x >> 5] = l1;
    red[2][threadIdx.x >> 5] = cep;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, c = 0.f, e = 0.f;
#pragma unroll
    for (int w = 0; w < NT / 32; ++w) {
      a += red[0][w];
      c += red[1][w];
      e += red[2][w];
    }
    float* o = terms + (long long)b * 3 * ws_frames + fr;
    o[0] = sqrtf(a / (float)(M + 1));
    o[ws_frames] = c / (float)n_mels;
    o[2LL * ws_frames] = kMcdScale * sqrtf(2.f * e);
  }
}

// out[b][j] = mean over the item's len_b / hop + 1 frames of terms[b][j]; four partial sums per thread, then
// block_sum_1024, in a fixed order (logdet_accumulate_varlen_kernel's pattern)
__global__ void __launch_bounds__(1024) spectral_distance_reduce_kernel(const float* __restrict__ terms, int ws_frames,
                                                                        const int* __restrict__ lengths, int T, int hop,
                                                                        float* __restrict__ out) {
  __shared__ float red[32];
  const int b = blockIdx.x;
  const int n = (lengths != nullptr ? lengths[b] : T) / hop + 1;
#pragma unroll 1
  for (int j = 0; j < 3; ++j) {
    const float* p = terms + ((long long)b * 3 + j) * ws_frames;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    int i = threadIdx.x;
    for (; i + 3 * 1024 < n; i += 4 * 1024) {
      s0 += p[i]; s1 += p[i + 1024]; s2 += p[i + 2048]; s3 += p[i + 3072];
    }
    for (; i < n; i += 1024) s0 += p[i];
    const float s = block_sum_1024((s0 + s1) + (s2 + s3), red);
    if (threadIdx.x == 0) out[(long long)b * 3 + j] = s / (float)n;
  }
}

}  // namespace cmwg

using namespace cmwg;

extern "C" size_t cmwg_spectral_distance_workspace_bytes(int B, int T, int n_fft, int hop) {
  if (B <= 0 || T <= 0 || n_fft <= 0 || hop <= 0) return 0;
  return (size_t)B * 3 * (size_t)(T / hop + 1) * sizeof(float);
}

extern "C" int cmwg_spectral_distance(const float* ref, const float* est, long long bstride, int B, int T,
                                      const int* lengths_host, const int* lengths_dev, const float* window,
                                      const float* fbt, const int* fb_lo, const int* fb_hi, const float* dct, int n_fft,
                                      int hop, int n_mels, int n_cep, void* workspace, float* out, void* stream) {
  if (!(n_fft >= 128 && n_fft <= 4096 && (n_fft & (n_fft - 1)) == 0)) {
    set_error("spectral_distance: n_fft must be a power of two in [128, 4096], got %d", n_fft);
    return CMWG_ERR_UNSUPPORTED;
  }
  CMWG_REQUIRE(B >= 0 && B <= 65535 && T >= 0 && hop > 0, "spectral_distance: bad sizes B=%d T=%d hop=%d", B, T, hop);
  // the log-mel difference sits in dynamic shared memory next to the FFT's < 44 KB
  CMWG_REQUIRE(n_mels >= 1 && n_mels <= 16384, "spectral_distance: n_mels must be in [1, 16384], got %d", n_mels);
  CMWG_REQUIRE(n_cep >= 2 && n_cep <= n_mels, "spectral_distance: n_cepstra must be in [2, n_mels = %d], got %d", n_mels,
               n_cep);
  CMWG_REQUIRE((lengths_host == nullptr) == (lengths_dev == nullptr),
               "spectral_distance: pass lengths both on the host and on the device, or neither");
  if (B == 0) return CMWG_OK;
  CMWG_REQUIRE(B == 1 || bstride >= T, "spectral_distance: batch stride %lld < T=%d", bstride, T);
  int max_len = T;
  if (lengths_host != nullptr) {
    max_len = 0;
    for (int b = 0; b < B; ++b) {
      CMWG_REQUIRE(lengths_host[b] > n_fft / 2 && lengths_host[b] <= T,
                   "spectral_distance: length %d of item %d outside (n_fft/2 = %d, T = %d]", lengths_host[b], b,
                   n_fft / 2, T);
      max_len = lengths_host[b] > max_len ? lengths_host[b] : max_len;
    }
  } else {
    CMWG_REQUIRE(T > n_fft / 2, "spectral_distance: length T=%d outside (n_fft/2 = %d, T]", T, n_fft / 2);
  }
  CMWG_REQUIRE(ref != nullptr && est != nullptr && window != nullptr && fbt != nullptr && fb_lo != nullptr &&
                   fb_hi != nullptr && dct != nullptr && workspace != nullptr && out != nullptr,
               "spectral_distance: NULL pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int ws_frames = T / hop + 1;
  float* terms = static_cast<float*>(workspace);
  const dim3 grid((unsigned)(max_len / hop + 1), (unsigned)B);
  const size_t dyn = (size_t)n_mels * sizeof(float);
#define CMWG_SD_CASE(N)                                                                                               \
  case N:                                                                                                             \
    if (dyn > 4096) /* past the 48 KB that needs no opt-in */                                                         \
      CMWG_CHECK_CUDA(cudaFuncSetAttribute(spectral_distance_frames_kernel<N>,                                       \
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));                    \
    spectral_distance_frames_kernel<N><<<grid, 256, dyn, st>>>(ref, est, bstride, T, lengths_dev, window, fbt, fb_lo,  \
                                                               fb_hi, dct, hop, n_mels, n_cep, ws_frames, terms);    \
    break;
  switch (n_fft) {
    CMWG_SD_CASE(128)
    CMWG_SD_CASE(256)
    CMWG_SD_CASE(512)
    CMWG_SD_CASE(1024)
    CMWG_SD_CASE(2048)
    CMWG_SD_CASE(4096)
  }
#undef CMWG_SD_CASE
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  spectral_distance_reduce_kernel<<<B, 1024, 0, st>>>(terms, ws_frames, lengths_dev, T, hop, out);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}
