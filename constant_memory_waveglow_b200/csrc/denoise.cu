// Bias-spectrum denoiser for synthesised audio (the `Denoiser` of NVIDIA's WaveGlow, mode 'zeros'): per item of a padded
// batch, STFT (n_fft, hop, window, center=True, reflect padding at the ITEM's end) -> |S| - strength * bias clamped at 0,
// phase kept -> inverse STFT (window-square normalised overlap-add) over the item's own samples.
//
// Two kernels.  denoise_frames_kernel: one CTA per (item, frame); the reflect-padded, windowed frame is transformed, its
// bins rescaled and transformed back in shared memory (fft.cuh), and the windowed time-domain frame is written to a
// (B, frames, n_fft) fp32 workspace -- the complex spectrogram never reaches HBM.  overlap_add_kernel: a thread per output
// sample sums the <= n_fft/hop frames that cover it in ascending frame order (no atomics: bitwise reproducible) and divides
// by the window-square envelope of the same frames.  Nothing an item's output depends on is read from another item or from
// beyond its own length, so a batched item is bit-identical to the same item run alone.
#include "fft.cuh"

namespace cmwg {

// X * max(|X| - strength * bias, 0) / |X|, and 0 where |X| = 0
__device__ __forceinline__ float2 subtract_bias(float2 X, float bias, float strength) {
  const float mag = sqrtf(fmaf(X.x, X.x, X.y * X.y));
  const float g = mag > 0.f ? fmaxf(mag - strength * bias, 0.f) / mag : 0.f;
  return make_float2(X.x * g, X.y * g);
}

// mag == NULL: denoise every frame fr = blockIdx.x < len_b / hop + 1 of item b = blockIdx.y into
//   frames_out[b][fr][0, NFFT) = window * irfft(subtract_bias(rfft(window * frame)));
// mag != NULL: one CTA writes mag[k] = |rfft(window * frame mag_frame)[k]|, k <= NFFT/2, of item 0 and returns.
template <int NFFT>
__global__ void __launch_bounds__(256) denoise_frames_kernel(const float* __restrict__ x, long long x_bstride, int T,
                                                             const int* __restrict__ lengths, const float* __restrict__ window,
                                                             const float* __restrict__ bias_mag, float strength, int hop,
                                                             int ws_frames, float* __restrict__ frames_out, int mag_frame,
                                                             float* __restrict__ mag) {
  using S = FftShape<NFFT>;
  constexpr int M = S::M, NT = 256;
  constexpr int PAIRS = M / 2 + 1;                 // bin pairs (k, M - k), k <= M/2
  constexpr int IT = (PAIRS + NT - 1) / NT;
  __shared__ float2 z[S::MP];
  __shared__ float2 tw[S::MP];

  const int b = blockIdx.y;
  const int fr = mag != nullptr ? mag_frame : (int)blockIdx.x;
  const int len = lengths != nullptr ? lengths[b] : T;
  if (fr > len / hop) return;                     // the item has len / hop + 1 frames
  const float* xb = x + (long long)b * x_bstride;
  const int start = fr * hop - NFFT / 2;

  fft_twiddles<NFFT, NT>(tw);
  for (int n = threadIdx.x; n < M; n += NT) {
    int i0 = reflect_index(start + 2 * n, len), i1 = reflect_index(start + 2 * n + 1, len);
    z[fft_bitrev_slot<NFFT>(n)] = make_float2(xb[i0] * window[2 * n], xb[i1] * window[2 * n + 1]);
  }
  __syncthreads();
  fft_radix2<NFFT, NT>(z, tw);

  // bins k and M - k come from the same two FFT outputs and feed the same two merged inputs of the inverse, so a thread
  // handles both and keeps them in registers across the barrier that frees z
  float2 zk[IT], zm[IT];
#pragma unroll
  for (int it = 0; it < IT; ++it) {
    const int k = threadIdx.x + it * NT;
    if (k >= PAIRS) continue;
    const float2 a = z[fft_padi(k & (M - 1))], c = z[fft_padi((M - k) & (M - 1))];
    float2 Xk = rfft_split(a, c, fft_split_twiddle<NFFT>(tw, k));
    float2 Xm = rfft_split(c, a, fft_split_twiddle<NFFT>(tw, M - k));
    if (mag != nullptr) {
      mag[k] = sqrtf(fmaf(Xk.x, Xk.x, Xk.y * Xk.y));
      mag[M - k] = sqrtf(fmaf(Xm.x, Xm.x, Xm.y * Xm.y));
      continue;
    }
    Xk = subtract_bias(Xk, bias_mag[k], strength);
    Xm = subtract_bias(Xm, bias_mag[M - k], strength);
    zk[it] = irfft_merge_conj(Xk, Xm, tw[fft_padi(k)]);
    if (k > 0) zm[it] = irfft_merge_conj(Xm, Xk, tw[fft_padi(M - k)]);
  }
  if (mag != nullptr) return;
  __syncthreads();
#pragma unroll
  for (int it = 0; it < IT; ++it) {
    const int k = threadIdx.x + it * NT;
    if (k >= PAIRS) continue;
    z[fft_bitrev_slot<NFFT>(k)] = zk[it];
    if (k > 0 && k < M / 2) z[fft_bitrev_slot<NFFT>(M - k)] = zm[it];
  }
  __syncthreads();
  fft_radix2<NFFT, NT>(z, tw);

  constexpr float inv_n = 1.f / (float)NFFT;      // a power of two: the scaling is exact
  float2* fo = reinterpret_cast<float2*>(frames_out + ((long long)b * ws_frames + fr) * NFFT);
  for (int n = threadIdx.x; n < M; n += NT) {
    const float2 F = z[fft_padi(n)];
    fo[n] = make_float2(F.x * inv_n * window[2 * n], -F.y * inv_n * window[2 * n + 1]);
  }
}

// out[b][t] = sum_f frames[b][f][p - f hop] / sum_f window[p - f hop]^2 over the frames f < len_b / hop + 1 that cover
// p = t + n_fft/2, in ascending f, for t < len_b; 0 for len_b <= t < T
__global__ void __launch_bounds__(256) overlap_add_kernel(const float* __restrict__ frames, int ws_frames,
                                                          const int* __restrict__ lengths, int T,
                                                          const float* __restrict__ window, int n_fft, int hop,
                                                          float* __restrict__ out) {
  const int b = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const int len = lengths != nullptr ? lengths[b] : T;
  float* o = out + (long long)b * T;
  if (t >= len) {
    o[t] = 0.f;
    return;
  }
  const int p = t + n_fft / 2;
  const int f_hi = min(p / hop, len / hop);
  const int f_lo = p - n_fft + 1 <= 0 ? 0 : (p - n_fft + hop) / hop;
  // sample j = p - f hop of frame f; the next frame's sample sits n_fft - hop further on
  int j = p - f_lo * hop;
  const float* fp = frames + ((long long)b * ws_frames + f_lo) * n_fft + j;
  float acc = 0.f, env = 0.f;
  for (int f = f_lo; f <= f_hi; ++f, j -= hop, fp += n_fft - hop) {
    const float w = window[j];
    acc += *fp;
    env = fmaf(w, w, env);
  }
  o[t] = acc / env;
}

static int check_stft_shape(const char* what, int n_fft, int hop) {
  CMWG_REQUIRE(n_fft >= 128 && n_fft <= 4096 && (n_fft & (n_fft - 1)) == 0,
               "%s: n_fft must be a power of two in [128, 4096], got %d", what, n_fft);
  CMWG_REQUIRE(hop > 0 && hop <= n_fft / 2, "%s: hop must be in [1, n_fft/2 = %d], got %d", what, n_fft / 2, hop);
  return CMWG_OK;
}

static int launch_frames(int n_fft, dim3 grid, cudaStream_t st, const float* x, long long x_bstride, int T, const int* lengths,
                  const float* window, const float* bias_mag, float strength, int hop, int ws_frames, float* frames_out,
                  int mag_frame, float* mag) {
#define CMWG_DN_CASE(N)                                                                                               \
  case N:                                                                                                             \
    denoise_frames_kernel<N><<<grid, 256, 0, st>>>(x, x_bstride, T, lengths, window, bias_mag, strength, hop, ws_frames, \
                                                    frames_out, mag_frame, mag);                                     \
    break;
  switch (n_fft) {
    CMWG_DN_CASE(128)
    CMWG_DN_CASE(256)
    CMWG_DN_CASE(512)
    CMWG_DN_CASE(1024)
    CMWG_DN_CASE(2048)
    CMWG_DN_CASE(4096)
    default:
      set_error("denoise: n_fft must be a power of two in [128, 4096], got %d", n_fft);
      return CMWG_ERR_ARG;
  }
#undef CMWG_DN_CASE
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

}  // namespace cmwg

using namespace cmwg;

extern "C" size_t cmwg_denoise_workspace_bytes(int B, int T, int n_fft, int hop) {
  if (B <= 0 || T <= 0 || n_fft <= 0 || hop <= 0) return 0;
  return (size_t)B * (size_t)(T / hop + 1) * (size_t)n_fft * sizeof(float);
}

extern "C" int cmwg_stft_frame_magnitude(const float* x, int T, const float* window, int n_fft, int hop, int frame,
                                         float* mag, void* stream) {
  CMWG_PROPAGATE(check_stft_shape("stft_frame_magnitude", n_fft, hop));
  CMWG_REQUIRE(T > n_fft / 2, "stft_frame_magnitude: reflect padding by n_fft/2 = %d needs more samples, got T=%d",
               n_fft / 2, T);
  CMWG_REQUIRE(frame >= 0 && frame <= T / hop, "stft_frame_magnitude: frame %d outside [0, %d]", frame, T / hop);
  CMWG_REQUIRE(x != nullptr && window != nullptr && mag != nullptr, "stft_frame_magnitude: NULL pointer");
  return launch_frames(n_fft, dim3(1, 1), (cudaStream_t)stream, x, T, T, nullptr, window, nullptr, 0.f, hop, 0, nullptr,
                       frame, mag);
}

extern "C" int cmwg_denoise(const float* x, long long x_bstride, int B, int T, const int* lengths_host, const int* lengths_dev,
                            const float* window, const float* bias_mag, float strength, int n_fft, int hop, void* workspace,
                            float* out, void* stream) {
  CMWG_PROPAGATE(check_stft_shape("denoise", n_fft, hop));
  CMWG_REQUIRE(B >= 0 && B <= 65535 && T >= 0, "denoise: bad sizes B=%d T=%d", B, T);
  CMWG_REQUIRE(strength >= 0.f && strength <= 3.4e38f, "denoise: strength must be a finite number >= 0, got %g",
               (double)strength);
  CMWG_REQUIRE((lengths_host == nullptr) == (lengths_dev == nullptr),
               "denoise: pass lengths both on the host and on the device, or neither");
  if (B == 0) return CMWG_OK;
  CMWG_REQUIRE(B == 1 || x_bstride >= T, "denoise: batch stride %lld < T=%d", x_bstride, T);
  int max_len = T;
  if (lengths_host != nullptr) {
    max_len = 0;
    for (int b = 0; b < B; ++b) {
      CMWG_REQUIRE(lengths_host[b] > n_fft / 2 && lengths_host[b] <= T,
                   "denoise: length %d of item %d outside (n_fft/2 = %d, T = %d]", lengths_host[b], b, n_fft / 2, T);
      max_len = lengths_host[b] > max_len ? lengths_host[b] : max_len;
    }
  } else {
    CMWG_REQUIRE(T > n_fft / 2, "denoise: length T=%d outside (n_fft/2 = %d, T]", T, n_fft / 2);
  }
  CMWG_REQUIRE(x != nullptr && window != nullptr && bias_mag != nullptr && workspace != nullptr && out != nullptr,
               "denoise: NULL pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int ws_frames = T / hop + 1;
  float* frames = static_cast<float*>(workspace);
  CMWG_PROPAGATE(launch_frames(n_fft, dim3((unsigned)(max_len / hop + 1), (unsigned)B), st, x, x_bstride, T, lengths_dev,
                               window, bias_mag, strength, hop, ws_frames, frames, -1, nullptr));
  overlap_add_kernel<<<dim3((unsigned)ceil_div(T, 256), (unsigned)B), 256, 0, st>>>(frames, ws_frames, lengths_dev, T,
                                                                                      window, n_fft, hop, out);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}
