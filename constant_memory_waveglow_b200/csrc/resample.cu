// Band-limited resampling (torchaudio.functional.resample, sinc_interp_hann / sinc_interp_kaiser) over a padded batch
// with per-item lengths, as a polyphase filter that evaluates only the taps inside the window's support.
//
// With O = orig / gcd, N = new / gcd, output sample n = k N + j of item b is
//   y[b, n] = sum_{m < L} table[m][j] * x[b, k O + first[j] + m - w],   x[b, i] = 0 outside [0, len_b)
// for n < n_out_b = ceil(N len_b / O), and 0 for n_out_b <= n < T_out.  table (L, N) holds, for phase j, the taps of
// torchaudio's kernel row j from index first[j] on, padded with exact zeros to L; the host builds it (resample.py).
//
// One thread per output sample; the L products are summed in ascending m with fmaf, starting from -0 so that an identity
// table (orig == new: L = 1, table 1, first 0, w 0) copies x bit for bit.  No atomics and nothing read from another item or
// from past len_b: each item's output is a function of (x[b, :len_b], len_b) alone, computed by the same instructions in
// the same order whatever the batch, so a batched item equals its solo call bit for bit.
#include "common.cuh"

namespace cmwg {

// grid.x covers max_b n_out_b (host lengths); the stride loop writes the zero tail of [max_b n_out_b, T_out) as well
__global__ void __launch_bounds__(256) resample_kernel(const float* __restrict__ x, long long x_bstride,
                                                       const int* __restrict__ lengths, int T,
                                                       const float* __restrict__ table, const int* __restrict__ first,
                                                       int O, int N, int L, int w, float* __restrict__ y,
                                                       long long y_bstride, int T_out) {
  const int b = blockIdx.y;
  const int len = lengths != nullptr ? lengths[b] : T;
  const long long lim = (long long)N * len;                 // n < n_out_b  <=>  n O < N len_b
  const float* xb = x + (long long)b * x_bstride;
  float* yb = y + (long long)b * y_bstride;
  // the loop counter is 64-bit: n + stride may pass INT_MAX when T_out is close to it; inside the loop n < T_out fits an int
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long nn = (long long)blockIdx.x * blockDim.x + threadIdx.x; nn < T_out; nn += stride) {
    const int n = (int)nn;
    if ((long long)n * O >= lim) {
      yb[n] = 0.f;
      continue;
    }
    const int k = n / N, j = n - k * N;
    const int s = k * O + first[j] - w;                     // input index of tap m = 0
    const float* c = table + j;
    float acc = -0.f;
    if (s >= 0 && s + L <= len) {
#pragma unroll 4
      for (int m = 0; m < L; ++m) acc = fmaf(c[(long long)m * N], xb[s + m], acc);
    } else {
#pragma unroll 4
      for (int m = 0; m < L; ++m) {
        const int i = s + m;
        acc = fmaf(c[(long long)m * N], (i >= 0 && i < len) ? xb[i] : 0.f, acc);
      }
    }
    yb[n] = acc;
  }
}

}  // namespace cmwg

using namespace cmwg;

extern "C" int cmwg_resample(const float* x, long long x_bstride, int B, int T, const int* lengths_host,
                             const int* lengths_dev, const float* table, const int* first, int O, int N, int L, int w,
                             float* y, long long y_bstride, int T_out, void* stream) {
  CMWG_REQUIRE(B >= 0 && B <= 65535 && T >= 0, "resample: bad sizes B=%d T=%d", B, T);
  CMWG_REQUIRE(O >= 1 && N >= 1 && L >= 1 && w >= 0, "resample: bad filter O=%d N=%d L=%d w=%d", O, N, L, w);
  const long long want = ((long long)N * T + O - 1) / O;
  CMWG_REQUIRE((long long)T_out == want, "resample: T_out=%d, expected ceil(N*T/O) = %lld", T_out, want);
  // k O + first[j] + m - w stays below T + 2 O + 2 w + L (first[j] < 2 w + O) and must fit an int
  CMWG_REQUIRE((long long)T + 2LL * O + 2LL * w + L < 2147483647LL, "resample: T=%d with O=%d, w=%d, L=%d overflows "
               "32-bit sample indices", T, O, w, L);
  CMWG_REQUIRE((lengths_host == nullptr) == (lengths_dev == nullptr),
               "resample: pass lengths both on the host and on the device, or neither");
  if (B == 0 || T_out == 0) return CMWG_OK;
  CMWG_REQUIRE(B == 1 || x_bstride >= T, "resample: batch stride %lld < T=%d", x_bstride, T);
  CMWG_REQUIRE(B == 1 || y_bstride >= T_out, "resample: output batch stride %lld < T_out=%d", y_bstride, T_out);
  int max_len = T;
  if (lengths_host != nullptr) {
    max_len = 0;
    for (int b = 0; b < B; ++b) {
      CMWG_REQUIRE(lengths_host[b] >= 1 && lengths_host[b] <= T, "resample: length %d of item %d outside [1, T = %d]",
                   lengths_host[b], b, T);
      max_len = lengths_host[b] > max_len ? lengths_host[b] : max_len;
    }
  }
  CMWG_REQUIRE(x != nullptr && table != nullptr && first != nullptr && y != nullptr, "resample: NULL pointer");
  const long long max_out = ((long long)N * max_len + O - 1) / O;
  const int blocks = (int)((max_out + 255) / 256);
  resample_kernel<<<dim3((unsigned)(blocks > 0 ? blocks : 1), (unsigned)B), 256, 0, (cudaStream_t)stream>>>(
      x, x_bstride, lengths_dev, T, table, first, O, N, L, w, y, y_bstride, T_out);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}
