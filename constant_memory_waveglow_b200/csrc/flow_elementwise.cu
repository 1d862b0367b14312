// HBM-bound flow primitives: invertible 1x1 conv (apply / weight-gradient / tiny LU), affine
// coupling (apply / backward), squeeze, NLL loss, per-batch sums.  All fp32, coalesced along the
// time axis (NCL layout), vectorised 4-wide where alignment allows, deterministic reductions.
#include "common.cuh"

#include <math_constants.h>
#include <stdarg.h>
#include <stdlib.h>

#include <vector>

namespace cmwg {

// ------------------------------------------------------------------------------------------------
// library-wide state
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";
unsigned long long g_launch_count = 0;

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

struct ProfRec { cudaEvent_t a, b; int cls; };
static bool g_prof_on = false;
static std::vector<ProfRec> g_prof;
static std::vector<cudaEvent_t> g_prof_pool;
static cudaEvent_t prof_event() {
  if (!g_prof_pool.empty()) { cudaEvent_t e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
  cudaEvent_t e;
  cudaEventCreate(&e);
  return e;
}
void prof_begin(cudaStream_t st, int cls) {
  if (!g_prof_on) return;
  ProfRec r;
  r.a = prof_event(); r.b = prof_event(); r.cls = (cls >= 0 && cls < CMWG_KCLASS_COUNT) ? cls : CMWG_KCLASS_COUNT - 1;
  cudaEventRecord(r.a, st);
  g_prof.push_back(r);
}
void prof_end(cudaStream_t st) {
  if (!g_prof_on || g_prof.empty()) return;
  cudaEventRecord(g_prof.back().b, st);
}

bool pdl_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* v = getenv("CMWG_PDL");
    on = (v && v[0] == '0') ? 0 : 1;
  }
  return on != 0;
}

int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) n = 148;
  }
  return n;
}

// ------------------------------------------------------------------------------------------------
// 1x1 conv apply: z[b,o,t] = sum_i M[o][i] x[b,i,t]
// one thread = VEC consecutive time steps of one batch item, all channels in registers.
// algorithmic bytes: 2 * B*C*T*4 (read x, write z)
// ------------------------------------------------------------------------------------------------
template <int C, int VEC>
__global__ void __launch_bounds__(256) conv1x1_apply_kernel(const float* __restrict__ w, int transpose_w,
                                                            const float* __restrict__ x, long long x_bs,
                                                            float* __restrict__ z, long long z_bs, int T,
                                                            int n_vec_per_batch, long long total) {
  __shared__ float ws[C * C];
  for (int i = threadIdx.x; i < C * C; i += blockDim.x) {
    int o = i / C, k = i % C;
    ws[i] = transpose_w ? w[k * C + o] : w[i];
  }
  __syncthreads();
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    int b = (int)(idx / n_vec_per_batch);
    int t = (int)(idx % n_vec_per_batch) * VEC;
    const float* xp = x + b * x_bs + t;
    float* zp = z + b * z_bs + t;
    float xv[C][VEC];
#pragma unroll
    for (int i = 0; i < C; ++i) {
      if (VEC == 4) {
        float4 v = *reinterpret_cast<const float4*>(xp + (long long)i * T);
        xv[i][0] = v.x; xv[i][1 % VEC] = v.y; xv[i][2 % VEC] = v.z; xv[i][3 % VEC] = v.w;
      } else {
        xv[i][0] = xp[(long long)i * T];
      }
    }
#pragma unroll
    for (int o = 0; o < C; ++o) {
      float acc[VEC];
#pragma unroll
      for (int v = 0; v < VEC; ++v) acc[v] = 0.f;
#pragma unroll
      for (int i = 0; i < C; ++i) {
        float wv = ws[o * C + i];
#pragma unroll
        for (int v = 0; v < VEC; ++v) acc[v] = fmaf(wv, xv[i][v], acc[v]);
      }
      if (VEC == 4) {
        *reinterpret_cast<float4*>(zp + (long long)o * T) = make_float4(acc[0], acc[1 % VEC], acc[2 % VEC], acc[3 % VEC]);
      } else {
        zp[(long long)o * T] = acc[0];
      }
    }
  }
}

// generic channel count (C <= 64): x column staged through shared memory
__global__ void __launch_bounds__(128) conv1x1_apply_generic_kernel(const float* __restrict__ w, int transpose_w,
                                                                    const float* __restrict__ x, long long x_bs,
                                                                    float* __restrict__ z, long long z_bs, int C,
                                                                    int T, int tiles_per_batch) {
  extern __shared__ float sm[];
  float* ws = sm;               // C*C
  float* xs = sm + C * C;       // C * 128
  for (int i = threadIdx.x; i < C * C; i += blockDim.x) {
    int o = i / C, k = i % C;
    ws[i] = transpose_w ? w[k * C + o] : w[i];
  }
  int b = blockIdx.x / tiles_per_batch;
  int t = (blockIdx.x % tiles_per_batch) * 128 + threadIdx.x;
  bool ok = t < T;
  for (int i = 0; i < C; ++i) xs[i * 128 + threadIdx.x] = ok ? x[b * x_bs + (long long)i * T + t] : 0.f;
  __syncthreads();
  if (!ok) return;
  for (int o = 0; o < C; ++o) {
    float acc = 0.f;
    for (int i = 0; i < C; ++i) acc = fmaf(ws[o * C + i], xs[i * 128 + threadIdx.x], acc);
    z[b * z_bs + (long long)o * T + t] = acc;
  }
}

template <int C>
static int launch_conv1x1_apply(const float* w, int tr, const float* x, long long x_bs, float* z, long long z_bs,
                                int B, int T, cudaStream_t st) {
  // 4-wide columns only while all C*4 inputs + accumulators stay in registers
  bool vec = (C <= 8) && (T % 4 == 0) && (x_bs % 4 == 0) && (z_bs % 4 == 0) && (((uintptr_t)x & 15) == 0) &&
             (((uintptr_t)z & 15) == 0);
  bool done = false;
  if constexpr (C <= 8) {
    if (vec) {
      int nv = T / 4;
      long long total = (long long)B * nv;
      int blocks = (int)std::min<long long>(ceil_div_ll(total, 256), (long long)num_sms() * 8);
      conv1x1_apply_kernel<C, 4><<<blocks, 256, 0, st>>>(w, tr, x, x_bs, z, z_bs, T, nv, total);
      done = true;
    }
  }
  if (!done) {
    long long total = (long long)B * T;
    int blocks = (int)std::min<long long>(ceil_div_ll(total, 256), (long long)num_sms() * 8);
    conv1x1_apply_kernel<C, 1><<<blocks, 256, 0, st>>>(w, tr, x, x_bs, z, z_bs, T, T, total);
  }
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

// ------------------------------------------------------------------------------------------------
// 1x1 conv weight gradient: dm[o][i] = sum_{b,t} dz[b,o,t] x[b,i,t]
// pass 1: each block reduces a (batch, 512-column) chunk into C*C partials; pass 2: fixed-order sum.
// ------------------------------------------------------------------------------------------------
// columns per block: 512 up to C = 32, 128 above (shared memory holds 2 * C * (cols + 1) floats)
static inline int wg_cols(int C) { return C <= 32 ? 512 : 128; }
constexpr int WG_THREADS = 256;

__global__ void __launch_bounds__(WG_THREADS) conv1x1_wgrad_partial_kernel(const float* __restrict__ dz,
                                                                            long long dz_bs,
                                                                            const float* __restrict__ x,
                                                                            long long x_bs, int C, int T,
                                                                            int chunks_per_batch, int WG_COLS,
                                                                            float* __restrict__ partial) {
  extern __shared__ float sm[];
  const int LD = WG_COLS + 1;
  float* dzs = sm;           // C * LD
  float* xs = sm + C * LD;   // C * LD
  float* red = xs + C * LD;  // WG_THREADS
  int b = blockIdx.x / chunks_per_batch;
  int t0 = (blockIdx.x % chunks_per_batch) * WG_COLS;
  int ncol = min(WG_COLS, T - t0);
  for (int idx = threadIdx.x; idx < C * WG_COLS; idx += WG_THREADS) {
    int c = idx / WG_COLS, k = idx % WG_COLS;
    bool ok = k < ncol;
    dzs[c * LD + k] = ok ? dz[b * dz_bs + (long long)c * T + t0 + k] : 0.f;
    xs[c * LD + k] = ok ? x[b * x_bs + (long long)c * T + t0 + k] : 0.f;
  }
  __syncthreads();
  const int P = C * C;
  float* out = partial + (long long)blockIdx.x * P;
  if (P >= WG_THREADS) {
    for (int p = threadIdx.x; p < P; p += WG_THREADS) {
      int o = p / C, i = p % C;
      float acc = 0.f;
      for (int k = 0; k < WG_COLS; ++k) acc = fmaf(dzs[o * LD + k], xs[i * LD + k], acc);
      out[p] = acc;
    }
  } else {
    int G = WG_THREADS / P;  // column groups per pair
    int p = threadIdx.x / G, g = threadIdx.x % G;
    float acc = 0.f;
    if (p < P) {
      int o = p / C, i = p % C;
      for (int k = g; k < WG_COLS; k += G) acc = fmaf(dzs[o * LD + k], xs[i * LD + k], acc);
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    if (p < P && g == 0) {
      float s = 0.f;
      for (int j = 0; j < G; ++j) s += red[p * G + j];
      out[p] = s;
    }
  }
}

__global__ void reduce_partials_kernel(const float* __restrict__ partial, int nblocks, int P, float* __restrict__ out) {
  int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  // pairwise-free fixed order: double accumulator keeps the cross-block sum exact enough to be
  // insensitive to the number of blocks
  double s = 0.0;
  for (int j = 0; j < nblocks; ++j) s += (double)partial[(long long)j * P + p];
  out[p] = (float)s;
}

__global__ void conv1x1_dw_finalize_kernel(const float* __restrict__ dm, const float* __restrict__ winv,
                                           const float* __restrict__ dlogdet, int c, int T, int inverse_mode,
                                           float* __restrict__ dw) {
  extern __shared__ float sm[];
  float* tmp = sm;  // c*c
  float scale = (*dlogdet) * (float)T;
  int n = c * c;
  if (!inverse_mode) {
    for (int p = threadIdx.x; p < n; p += blockDim.x) {
      int o = p / c, i = p % c;
      dw[p] = dm[p] + winv[i * c + o] * scale;  // W^-T[o][i] = winv[i][o]
    }
    return;
  }
  // tmp = W^-T dm : tmp[o][i] = sum_k winv[k][o] dm[k][i]
  for (int p = threadIdx.x; p < n; p += blockDim.x) {
    int o = p / c, i = p % c;
    float s = 0.f;
    for (int k = 0; k < c; ++k) s = fmaf(winv[k * c + o], dm[k * c + i], s);
    tmp[p] = s;
  }
  __syncthreads();
  // dw = -(tmp W^-T) - W^-T scale : (tmp W^-T)[o][i] = sum_k tmp[o][k] winv[i][k]
  for (int p = threadIdx.x; p < n; p += blockDim.x) {
    int o = p / c, i = p % c;
    float s = 0.f;
    for (int k = 0; k < c; ++k) s = fmaf(tmp[o * c + k], winv[i * c + k], s);
    dw[p] = -s - winv[i * c + o] * scale;
  }
}

// ------------------------------------------------------------------------------------------------
// Whole backward of the invertible 1x1 conv in two launches (C <= 8):
//   pass 1, one sweep over (out, dout):  in = Minv out  (the freed input, re-materialised: efficient_modules.py:236,268),
//           din = Mt dout (:239,273), block partials of dm[o][i] = sum dout[o] in[i] (:240-241,274-275);
//   pass 2, one CTA: fixed-order sum of the block partials + the dW formula of conv1x1_dw_finalize_kernel.
// One thread owns 4 consecutive time steps of one batch item with every channel in registers; the C*C outer-product
// accumulators stay in registers across the grid-stride loop and are folded once per CTA (shuffles, then warp order).
// ------------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(256) conv1x1_bwd_fused_kernel(const float* __restrict__ minv, const float* __restrict__ w,
                                                                int transpose_w, const float* __restrict__ out, long long out_bs,
                                                                const float* __restrict__ dout, long long dout_bs,
                                                                float* __restrict__ restored, long long r_bs,
                                                                float* __restrict__ din, long long din_bs, int T, int nv,
                                                                long long total, float* __restrict__ partial) {
  __shared__ float m1[C * C], m2[C * C];
  __shared__ float red[8][C * C];
  for (int i = threadIdx.x; i < C * C; i += 256) {
    const int o = i / C, k = i % C;
    m1[i] = minv[i];
    m2[i] = transpose_w ? w[k * C + o] : w[i];
  }
  __syncthreads();
  float acc[C * C];
#pragma unroll
  for (int i = 0; i < C * C; ++i) acc[i] = 0.f;
  for (long long idx = blockIdx.x * 256ll + threadIdx.x; idx < total; idx += (long long)gridDim.x * 256) {
    const int b = (int)(idx / nv), t = (int)(idx % nv) * 4;
    float zv[C][4], gv[C][4], xv[C][4];
#pragma unroll
    for (int i = 0; i < C; ++i) {
      const float4 a = *reinterpret_cast<const float4*>(out + b * out_bs + (long long)i * T + t);
      const float4 g = *reinterpret_cast<const float4*>(dout + b * dout_bs + (long long)i * T + t);
      zv[i][0] = a.x; zv[i][1] = a.y; zv[i][2] = a.z; zv[i][3] = a.w;
      gv[i][0] = g.x; gv[i][1] = g.y; gv[i][2] = g.z; gv[i][3] = g.w;
    }
#pragma unroll
    for (int o = 0; o < C; ++o) {
      float x4[4] = {0.f, 0.f, 0.f, 0.f}, d4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int i = 0; i < C; ++i) {
        const float a = m1[o * C + i], bq = m2[o * C + i];
#pragma unroll
        for (int v = 0; v < 4; ++v) { x4[v] = fmaf(a, zv[i][v], x4[v]); d4[v] = fmaf(bq, gv[i][v], d4[v]); }
      }
#pragma unroll
      for (int v = 0; v < 4; ++v) xv[o][v] = x4[v];
      if (restored) *reinterpret_cast<float4*>(restored + b * r_bs + (long long)o * T + t) = make_float4(x4[0], x4[1], x4[2], x4[3]);
      *reinterpret_cast<float4*>(din + b * din_bs + (long long)o * T + t) = make_float4(d4[0], d4[1], d4[2], d4[3]);
    }
    if (partial) {
#pragma unroll
      for (int o = 0; o < C; ++o)
#pragma unroll
        for (int i = 0; i < C; ++i)
#pragma unroll
          for (int v = 0; v < 4; ++v) acc[o * C + i] = fmaf(gv[o][v], xv[i][v], acc[o * C + i]);
    }
  }
  if (!partial) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < C * C; ++i) {
    const float v = warp_sum(acc[i]);
    if (lane == 0) red[warp][i] = v;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C * C; i += 256) {
    float sacc = 0.f;
#pragma unroll
    for (int wq = 0; wq < 8; ++wq) sacc += red[wq][i];
    partial[(long long)blockIdx.x * C * C + i] = sacc;
  }
}

// pass 2: dm = sum_j partial[j] (fixed order, fp64), then dW as in conv1x1_dw_finalize_kernel
__global__ void __launch_bounds__(64) conv1x1_dw_from_partials_kernel(const float* __restrict__ partial, int nblocks,
                                                                      const float* __restrict__ winv,
                                                                      const float* __restrict__ dlogdet, int c, int T,
                                                                      int inverse_mode, float* __restrict__ dw) {
  __shared__ float dm[64], tmp[64];
  const int n = c * c;
  const float scale = (dlogdet ? *dlogdet : 0.f) * (float)T;
  for (int p = threadIdx.x; p < n; p += 64) {
    double sacc = 0.0;
    for (int j = 0; j < nblocks; ++j) sacc += (double)partial[(long long)j * n + p];
    dm[p] = (float)sacc;
  }
  __syncthreads();
  if (!inverse_mode) {
    for (int p = threadIdx.x; p < n; p += 64) {
      const int o = p / c, i = p % c;
      dw[p] = dm[p] + winv[i * c + o] * scale;
    }
    return;
  }
  for (int p = threadIdx.x; p < n; p += 64) {
    const int o = p / c, i = p % c;
    float sacc = 0.f;
    for (int k = 0; k < c; ++k) sacc = fmaf(winv[k * c + o], dm[k * c + i], sacc);
    tmp[p] = sacc;
  }
  __syncthreads();
  for (int p = threadIdx.x; p < n; p += 64) {
    const int o = p / c, i = p % c;
    float sacc = 0.f;
    for (int k = 0; k < c; ++k) sacc = fmaf(tmp[o * c + k], winv[i * c + k], sacc);
    dw[p] = -sacc - winv[i * c + o] * scale;
  }
}

template <int C>
static int launch_conv1x1_bwd_fused(const float* minv, const float* w, int tr, const float* out, long long out_bs,
                                    const float* dout, long long dout_bs, float* restored, long long r_bs, float* din,
                                    long long din_bs, int B, int T, float* partial, int blocks, cudaStream_t st) {
  const int nv = T / 4;
  conv1x1_bwd_fused_kernel<C><<<blocks, 256, 0, st>>>(minv, w, tr, out, out_bs, dout, dout_bs, restored, r_bs, din, din_bs, T,
                                                       nv, (long long)B * nv, partial);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

// ------------------------------------------------------------------------------------------------
// tiny LU (Gauss-Jordan with partial pivoting, fp64 internally): inverse + log det, c <= 64
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(64) small_inverse_logdet_kernel(const float* __restrict__ w, int c,
                                                                  float* __restrict__ winv,
                                                                  float* __restrict__ logdet) {
  extern __shared__ double smd[];
  const int LD = 2 * c;
  double* a = smd;  // c x 2c augmented [W | I]
  __shared__ int piv_row;
  __shared__ double s_logabs;
  __shared__ int s_sign;
  int r = threadIdx.x;
  if (r < c) {
    for (int j = 0; j < c; ++j) {
      a[r * LD + j] = (double)w[r * c + j];
      a[r * LD + c + j] = (r == j) ? 1.0 : 0.0;
    }
  }
  if (r == 0) { s_logabs = 0.0; s_sign = 1; }
  __syncthreads();
  for (int k = 0; k < c; ++k) {
    if (r == 0) {
      int best = k;
      double bv = fabs(a[k * LD + k]);
      for (int i = k + 1; i < c; ++i) {
        double v = fabs(a[i * LD + k]);
        if (v > bv) { bv = v; best = i; }
      }
      piv_row = best;
    }
    __syncthreads();
    int pr = piv_row;
    if (pr != k) {
      for (int j = r; j < LD; j += blockDim.x) {
        double tmp = a[k * LD + j];
        a[k * LD + j] = a[pr * LD + j];
        a[pr * LD + j] = tmp;
      }
    }
    __syncthreads();
    double pv = a[k * LD + k];
    if (r == 0) {
      if (pr != k) s_sign = -s_sign;
      if (pv < 0) s_sign = -s_sign;
      s_logabs += log(fabs(pv));
    }
    __syncthreads();
    // scale pivot row
    for (int j = r; j < LD; j += blockDim.x) a[k * LD + j] /= pv;
    __syncthreads();
    if (r < c && r != k) {
      double f = a[r * LD + k];
      if (f != 0.0)
        for (int j = 0; j < LD; ++j) a[r * LD + j] -= f * a[k * LD + j];
    }
    __syncthreads();
  }
  if (r < c)
    for (int j = 0; j < c; ++j) winv[r * c + j] = (float)a[r * LD + c + j];
  if (r == 0) {
    // Tensor.logdet(): NaN for a negative determinant, -inf for a singular matrix
    float v = (float)s_logabs;
    if (s_sign < 0) v = CUDART_NAN_F;
    *logdet = v;
  }
}

// ------------------------------------------------------------------------------------------------
// affine coupling
// algorithmic bytes (fwd): (c + 2cin + c) * B*T*4  (read x and lst, write z)
// ------------------------------------------------------------------------------------------------
template <int VEC>
__global__ void __launch_bounds__(256) coupling_apply_kernel(const float* __restrict__ x, long long x_bs,
                                                             const float* __restrict__ lst,
                                                             float* __restrict__ z, long long z_bs,
                                                             float* __restrict__ neg_ls, int cin, int T,
                                                             int inverse, long long total,
                                                             const int* __restrict__ len = nullptr) {
  // len != nullptr: columns t >= len[b] of z and neg_ls are written as 0 (a select: the flow state there may be non-finite)
  // idx enumerates (b, j, t/VEC)
  int nv = T / VEC;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    int tv = (int)(idx % nv);
    int j = (int)((idx / nv) % cin);
    int b = (int)(idx / ((long long)nv * cin));
    long long t = (long long)tv * VEC;
    const float* xa = x + b * x_bs + (long long)j * T + t;
    const float* xb = xa + (long long)cin * T;
    const float* ls = lst + ((long long)b * 2 * cin + j) * T + t;
    const float* tt = ls + (long long)cin * T;
    float* za = z + b * z_bs + (long long)j * T + t;
    float* zb = za + (long long)cin * T;
    float a[VEC], bb[VEC], l[VEC], s[VEC], o[VEC], nl[VEC];
    if (VEC == 4) {
      float4 v;
      v = *reinterpret_cast<const float4*>(xa); a[0] = v.x; a[1 % VEC] = v.y; a[2 % VEC] = v.z; a[3 % VEC] = v.w;
      v = *reinterpret_cast<const float4*>(xb); bb[0] = v.x; bb[1 % VEC] = v.y; bb[2 % VEC] = v.z; bb[3 % VEC] = v.w;
      v = *reinterpret_cast<const float4*>(ls); l[0] = v.x; l[1 % VEC] = v.y; l[2 % VEC] = v.z; l[3 % VEC] = v.w;
      v = *reinterpret_cast<const float4*>(tt); s[0] = v.x; s[1 % VEC] = v.y; s[2 % VEC] = v.z; s[3 % VEC] = v.w;
    } else {
      a[0] = *xa; bb[0] = *xb; l[0] = *ls; s[0] = *tt;
    }
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      float e = expf(l[v]);
      o[v] = inverse ? (bb[v] - s[v]) / e : fmaf(bb[v], e, s[v]);
      nl[v] = -l[v];
    }
    if (len != nullptr) {
      const int lb = __ldg(len + b);
#pragma unroll
      for (int v = 0; v < VEC; ++v)
        if (t + v >= lb) a[v] = o[v] = nl[v] = 0.f;
    }
    if (VEC == 4) {
      *reinterpret_cast<float4*>(za) = make_float4(a[0], a[1 % VEC], a[2 % VEC], a[3 % VEC]);
      *reinterpret_cast<float4*>(zb) = make_float4(o[0], o[1 % VEC], o[2 % VEC], o[3 % VEC]);
      if (neg_ls)
        *reinterpret_cast<float4*>(neg_ls + ((long long)b * cin + j) * T + t) =
            make_float4(nl[0], nl[1 % VEC], nl[2 % VEC], nl[3 % VEC]);
    } else {
      *za = a[0];
      *zb = o[0];
      if (neg_ls) neg_ls[((long long)b * cin + j) * T + t] = nl[0];
    }
  }
}

// backward elementwise half; see cmwg_coupling_bwd in the header
__global__ void __launch_bounds__(256) coupling_bwd_kernel(const float* __restrict__ out, long long out_bs,
                                                           const float* __restrict__ lst,
                                                           const float* __restrict__ dout, long long dout_bs,
                                                           const float* __restrict__ dls, long long dls_bs,
                                                           float* __restrict__ restored,
                                                           float* __restrict__ dlst, float* __restrict__ din,
                                                           int cin, int T, int inverse, long long total) {
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    int t = (int)(idx % T);
    int j = (int)((idx / T) % cin);
    int b = (int)(idx / ((long long)T * cin));
    long long oa = b * out_bs + (long long)j * T + t;
    long long ob = oa + (long long)cin * T;
    long long la = ((long long)b * 2 * cin + j) * T + t;
    long long lb = la + (long long)cin * T;
    float ya = out[oa], yb = out[ob];
    float ls = lst[la], tt = lst[lb];
    float s = expf(ls);
    float ga = dout[b * dout_bs + (long long)j * T + t];
    float gb = dout[b * dout_bs + (long long)(cin + j) * T + t];
    float gl = dls[b * dls_bs + (long long)j * T + t];
    float in_b, g_ls, g_t, din_b;
    if (!inverse) {
      // forward call was zb = xb*s + t; outputs (z, log_s)
      in_b = (yb - tt) / s;            // xb
      g_ls = gb * in_b * s + gl;       // dzb*xb*s + dlog_s
      g_t = gb;
      din_b = gb * s;
    } else {
      // forward call was xb = (zb - t)/s; outputs (x, -log_s); yb = xb, incoming gl = d(-log_s)
      in_b = fmaf(yb, s, tt);          // zb
      g_ls = -gb * yb - gl;
      g_t = -gb / s;
      din_b = gb / s;
    }
    long long ra = ((long long)b * 2 * cin + j) * T + t;
    long long rb = ra + (long long)cin * T;
    restored[ra] = ya;
    restored[rb] = in_b;
    dlst[la] = g_ls;
    dlst[lb] = g_t;
    din[ra] = ga;
    din[rb] = din_b;
  }
}

// ------------------------------------------------------------------------------------------------
// squeeze / unsqueeze: (B, T) <-> (B, G, T/G); a transpose of a [T/G][G] matrix per batch item
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) squeeze_kernel(const float* __restrict__ x, float* __restrict__ out, int Tq,
                                                      int G, int inverse, long long total) {
  // forward: out[b][g][t] = x[b][t*G + g]; consecutive threads walk the OUTPUT
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    long long per = (long long)Tq * G;
    long long b = idx / per;
    long long r = idx % per;
    if (!inverse) {
      int g = (int)(r / Tq), t = (int)(r % Tq);
      out[idx] = x[b * per + (long long)t * G + g];
    } else {
      int t = (int)(r / G), g = (int)(r % G);
      out[idx] = x[b * per + (long long)g * Tq + t];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// reductions: per-batch sum, NLL loss
// ------------------------------------------------------------------------------------------------
__device__ float block_sum_1024(float v, float* red) {
  v = warp_sum(v);
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) red[wid] = v;
  __syncthreads();
  int nw = (blockDim.x + 31) >> 5;
  float r = (threadIdx.x < nw) ? red[threadIdx.x] : 0.f;
  if (wid == 0) r = warp_sum(r);
  __syncthreads();
  return r;  // valid in warp 0
}

__global__ void __launch_bounds__(1024) sum_per_batch_kernel(const float* __restrict__ a, long long a_bs, int N,
                                                             float* __restrict__ out, int accumulate,
                                                             float scale) {
  __shared__ float red[32];
  int b = blockIdx.x;
  const float* p = a + b * a_bs;
  // four independent partial sums per thread (fixed order: deterministic) keep 4 loads in flight
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  int i = threadIdx.x;
  for (; i + 3 * 1024 < N; i += 4 * 1024) {
    s0 += p[i]; s1 += p[i + 1024]; s2 += p[i + 2048]; s3 += p[i + 3072];
  }
  for (; i < N; i += 1024) s0 += p[i];
  float s = block_sum_1024((s0 + s1) + (s2 + s3), red);
  if (threadIdx.x == 0) out[b] = (accumulate ? out[b] : 0.f) + scale * s;
}

// logdet += log_det_W + log_s.sum((1, 2))  (model/waveglow.py:175,199) in one launch: out[b] = prev[b] + *ldw + sum a[b, :]
__global__ void __launch_bounds__(1024) logdet_accumulate_kernel(const float* __restrict__ a, long long a_bs, int N,
                                                                 const float* __restrict__ prev,
                                                                 const float* __restrict__ ldw, float* __restrict__ out) {
  __shared__ float red[32];
  const int b = blockIdx.x;
  const float* p = a + b * a_bs;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  int i = threadIdx.x;
  for (; i + 3 * 1024 < N; i += 4 * 1024) {
    s0 += p[i]; s1 += p[i + 1024]; s2 += p[i + 2048]; s3 += p[i + 3072];
  }
  for (; i < N; i += 1024) s0 += p[i];
  const float s = block_sum_1024((s0 + s1) + (s2 + s3), red);
  if (threadIdx.x == 0) out[b] = ((prev ? prev[b] : 0.f) + (ldw ? *ldw : 0.f)) + s;
}

// per-item lengths: out[b] = prev[b] + *ldw * len[b] + sum over channels c < C and columns t < len[b] of a[b, c, t].
// The valid (C, n) block is walked as the contiguous C * n tensor logdet_accumulate_kernel sums for the item alone, in the same
// order, and ldw * n is the `logdet * T` of that call: the result is bit-identical to it.
__global__ void __launch_bounds__(1024) logdet_accumulate_varlen_kernel(const float* __restrict__ a, long long a_bs, int C,
                                                                        int T, const int* __restrict__ len,
                                                                        const float* __restrict__ prev,
                                                                        const float* __restrict__ ldw, float* __restrict__ out) {
  __shared__ float red[32];
  const int b = blockIdx.x;
  const int n = min(max(len[b], 0), T);
  const int N = C * n;
  const float* p = a + b * a_bs;
  auto at = [&](int i) { const int c = i / n; return p[(long long)c * T + (i - c * n)]; };
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  int i = threadIdx.x;
  for (; i + 3 * 1024 < N; i += 4 * 1024) {
    s0 += at(i); s1 += at(i + 1024); s2 += at(i + 2048); s3 += at(i + 3072);
  }
  for (; i < N; i += 1024) s0 += at(i);
  const float s = block_sum_1024((s0 + s1) + (s2 + s3), red);
  if (threadIdx.x == 0) out[b] = ((prev ? prev[b] : 0.f) + (ldw ? *ldw * (float)n : 0.f)) + s;
}

__global__ void __launch_bounds__(1024) nll_rows_kernel(const float* __restrict__ z, int T, float* __restrict__ rows) {
  __shared__ float red[32];
  int b = blockIdx.x;
  const float* p = z + (long long)b * T;
  float s = 0.f;
  for (int i = threadIdx.x; i < T; i += blockDim.x) s = fmaf(p[i], p[i], s);
  s = block_sum_1024(s, red);
  if (threadIdx.x == 0) rows[b] = s;
}

__global__ void nll_final_kernel(const float* __restrict__ rows, const float* __restrict__ logdet, int B, int T,
                                 float inv_sigma2, int mean, float* __restrict__ loss) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    float s = 0.f;
    for (int b = 0; b < B; ++b) s += 0.5f * rows[b] * inv_sigma2 - logdet[b];
    s /= (float)B;
    if (mean) s /= (float)T;
    *loss = s;
  }
}

__global__ void __launch_bounds__(256) scale_kernel(const float* __restrict__ z, float* __restrict__ dz, float k,
                                                    long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    dz[i] = z[i] * k;
}

}  // namespace cmwg

using namespace cmwg;

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

const char* cmwg_last_error(void) { return g_err; }
int cmwg_version(void) { return 100; }
unsigned long long cmwg_launch_count(void) { return g_launch_count; }
void cmwg_reset_launch_count(void) { g_launch_count = 0; }

int cmwg_profile_enable(int on) {
  for (auto& r : g_prof) { g_prof_pool.push_back(r.a); g_prof_pool.push_back(r.b); }
  g_prof.clear();
  g_prof_on = on != 0;
  return CMWG_OK;
}

int cmwg_profile_collect(double* ms, long long* launches) {
  for (int i = 0; i < CMWG_KCLASS_COUNT; ++i) { ms[i] = 0.0; launches[i] = 0; }
  for (auto& r : g_prof) {
    CMWG_CHECK_CUDA(cudaEventSynchronize(r.b));
    float t = 0.f;
    CMWG_CHECK_CUDA(cudaEventElapsedTime(&t, r.a, r.b));
    ms[r.cls] += t;
    launches[r.cls] += 1;
    g_prof_pool.push_back(r.a);
    g_prof_pool.push_back(r.b);
  }
  g_prof.clear();
  return CMWG_OK;
}

int cmwg_small_inverse_logdet(const float* w, int c, float* w_inv, float* logdet, void* stream) {
  CMWG_REQUIRE(c >= 1 && c <= 64, "cmwg_small_inverse_logdet: c=%d out of range [1,64]", c);
  cudaStream_t st = (cudaStream_t)stream;
  size_t smem = (size_t)c * 2 * c * sizeof(double);
  if (smem > 48 * 1024)
    CMWG_CHECK_CUDA(cudaFuncSetAttribute(small_inverse_logdet_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem));
  small_inverse_logdet_kernel<<<1, 64, smem, st>>>(w, c, w_inv, logdet);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

int cmwg_conv1x1_apply(const float* w, int transpose_w, const float* x, long long x_bstride, float* z,
                       long long z_bstride, int B, int C, int T, void* stream) {
  CMWG_REQUIRE(C >= 1 && C <= 64, "cmwg_conv1x1_apply: C=%d out of range [1,64]", C);
  if (B == 0 || T == 0) return CMWG_OK;
  cudaStream_t st = (cudaStream_t)stream;
  switch (C) {
    case 2: return launch_conv1x1_apply<2>(w, transpose_w, x, x_bstride, z, z_bstride, B, T, st);
    case 4: return launch_conv1x1_apply<4>(w, transpose_w, x, x_bstride, z, z_bstride, B, T, st);
    case 6: return launch_conv1x1_apply<6>(w, transpose_w, x, x_bstride, z, z_bstride, B, T, st);
    case 8: return launch_conv1x1_apply<8>(w, transpose_w, x, x_bstride, z, z_bstride, B, T, st);
    case 12: return launch_conv1x1_apply<12>(w, transpose_w, x, x_bstride, z, z_bstride, B, T, st);
    case 14: return launch_conv1x1_apply<14>(w, transpose_w, x, x_bstride, z, z_bstride, B, T, st);
    case 16: return launch_conv1x1_apply<16>(w, transpose_w, x, x_bstride, z, z_bstride, B, T, st);
    default: break;
  }
  int tiles = ceil_div(T, 128);
  size_t smem = ((size_t)C * C + (size_t)C * 128) * sizeof(float);
  conv1x1_apply_generic_kernel<<<B * tiles, 128, smem, st>>>(w, transpose_w, x, x_bstride, z, z_bstride, C, T, tiles);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

size_t cmwg_conv1x1_wgrad_workspace(int B, int C, int T) {
  return (size_t)B * ceil_div(T, wg_cols(C)) * C * C * sizeof(float);
}

int cmwg_conv1x1_wgrad(const float* dz, long long dz_bstride, const float* x, long long x_bstride, int B, int C,
                       int T, float* dm, void* workspace, void* stream) {
  CMWG_REQUIRE(C >= 1 && C <= 128, "cmwg_conv1x1_wgrad: C=%d out of range [1,128]", C);
  cudaStream_t st = (cudaStream_t)stream;
  const int WG_COLS = wg_cols(C);
  int chunks = ceil_div(T, WG_COLS);
  int nblocks = B * chunks;
  size_t smem = ((size_t)2 * C * (WG_COLS + 1) + WG_THREADS) * sizeof(float);
  if (smem > 48 * 1024)
    CMWG_CHECK_CUDA(cudaFuncSetAttribute(conv1x1_wgrad_partial_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem));
  conv1x1_wgrad_partial_kernel<<<nblocks, WG_THREADS, smem, st>>>(dz, dz_bstride, x, x_bstride, C, T, chunks, WG_COLS,
                                                                  (float*)workspace);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  int P = C * C;
  reduce_partials_kernel<<<ceil_div(P, 128), 128, 0, st>>>((const float*)workspace, nblocks, P, dm);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

int cmwg_conv1x1_dw_finalize(const float* dm, const float* w_inv, const float* dlogdet, int c, int T,
                             int inverse_mode, float* dw, void* stream) {
  CMWG_REQUIRE(c >= 1 && c <= 64, "cmwg_conv1x1_dw_finalize: c=%d out of range [1,64]", c);
  conv1x1_dw_finalize_kernel<<<1, 256, (size_t)c * c * sizeof(float), (cudaStream_t)stream>>>(dm, w_inv, dlogdet, c, T,
                                                                                              inverse_mode, dw);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

static inline int conv1x1_bwd_blocks(int B, int T) {
  return (int)std::min<long long>(ceil_div_ll((long long)B * (T / 4), 256), (long long)num_sms() * 2);
}

size_t cmwg_conv1x1_backward_workspace(int B, int C, int T) {
  const size_t fused = (size_t)std::max(conv1x1_bwd_blocks(B, T), 1) * C * C * sizeof(float);
  return std::max(fused, cmwg_conv1x1_wgrad_workspace(B, C, T)) + (size_t)C * C * sizeof(float) + 256;
}

int cmwg_conv1x1_backward(const float* w, const float* w_inv, int inverse_mode, const float* out, long long out_bstride,
                          const float* dout, long long dout_bstride, const float* dlogdet, int B, int C, int T,
                          float* restored, long long restored_bstride, float* din, long long din_bstride, float* dw,
                          void* workspace, void* stream) {
  CMWG_REQUIRE(w && w_inv && out && dout && din, "cmwg_conv1x1_backward: null argument");
  CMWG_REQUIRE(C >= 1 && C <= 64, "cmwg_conv1x1_backward: C=%d out of range [1,64]", C);
  CMWG_REQUIRE(!dw || workspace, "cmwg_conv1x1_backward: the weight gradient needs a workspace");
  if (B == 0 || T == 0) return CMWG_OK;
  cudaStream_t st = (cudaStream_t)stream;
  // forward was out = M in with M = W (inverse_mode 0) or W^-1 (1):  in = M^-1 out,  din = M^T dout
  const float* m_restore = inverse_mode ? w : w_inv;
  const float* m_din = inverse_mode ? w_inv : w;
  auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  const bool fusable = C <= 8 && (C % 2 == 0) && T % 4 == 0 && out_bstride % 4 == 0 && dout_bstride % 4 == 0 &&
                       din_bstride % 4 == 0 && (!restored || restored_bstride % 4 == 0) && al16(out) && al16(dout) &&
                       al16(din) && (!restored || al16(restored));
  if (fusable) {
    const int blocks = conv1x1_bwd_blocks(B, T);
    float* partial = dw ? reinterpret_cast<float*>(workspace) : nullptr;
    int rc;
    switch (C) {
      case 2: rc = launch_conv1x1_bwd_fused<2>(m_restore, m_din, 1, out, out_bstride, dout, dout_bstride, restored, restored_bstride, din, din_bstride, B, T, partial, blocks, st); break;
      case 4: rc = launch_conv1x1_bwd_fused<4>(m_restore, m_din, 1, out, out_bstride, dout, dout_bstride, restored, restored_bstride, din, din_bstride, B, T, partial, blocks, st); break;
      case 6: rc = launch_conv1x1_bwd_fused<6>(m_restore, m_din, 1, out, out_bstride, dout, dout_bstride, restored, restored_bstride, din, din_bstride, B, T, partial, blocks, st); break;
      default: rc = launch_conv1x1_bwd_fused<8>(m_restore, m_din, 1, out, out_bstride, dout, dout_bstride, restored, restored_bstride, din, din_bstride, B, T, partial, blocks, st); break;
    }
    CMWG_PROPAGATE(rc);
    if (dw) {
      conv1x1_dw_from_partials_kernel<<<1, 64, 0, st>>>(partial, blocks, w_inv, dlogdet, C, T, inverse_mode, dw);
      CMWG_COUNT_LAUNCH();
      CMWG_LAUNCH_CHECK();
    }
    return CMWG_OK;
  }
  // general shapes: the separate kernels, same arithmetic
  float* scratch_in = restored;
  CMWG_REQUIRE(restored || !dw, "cmwg_conv1x1_backward: general shapes need `restored` to form the weight gradient");
  if (restored) CMWG_PROPAGATE(cmwg_conv1x1_apply(m_restore, 0, out, out_bstride, restored, restored_bstride, B, C, T, stream));
  CMWG_PROPAGATE(cmwg_conv1x1_apply(m_din, 1, dout, dout_bstride, din, din_bstride, B, C, T, stream));
  if (dw) {
    float* dm = reinterpret_cast<float*>(workspace);
    void* ws2 = reinterpret_cast<uint8_t*>(workspace) + align_up((size_t)C * C * sizeof(float), 256);
    CMWG_PROPAGATE(cmwg_conv1x1_wgrad(dout, dout_bstride, scratch_in, restored_bstride, B, C, T, dm, ws2, stream));
    CMWG_REQUIRE(dlogdet, "cmwg_conv1x1_backward: dlogdet missing");
    CMWG_PROPAGATE(cmwg_conv1x1_dw_finalize(dm, w_inv, dlogdet, C, T, inverse_mode, dw, stream));
  }
  return CMWG_OK;
}

int cmwg_coupling_apply(const float* x, long long x_bstride, const float* lst, float* z, long long z_bstride,
                        float* neg_log_s, int B, int cin, int T, int inverse, void* stream) {
  if (B == 0 || T == 0 || cin == 0) return CMWG_OK;
  cudaStream_t st = (cudaStream_t)stream;
  bool vec = (T % 4 == 0) && (x_bstride % 4 == 0) && (z_bstride % 4 == 0) && (((uintptr_t)x & 15) == 0) &&
             (((uintptr_t)z & 15) == 0) && (((uintptr_t)lst & 15) == 0) && (((uintptr_t)neg_log_s & 15) == 0);
  if (vec) {
    long long total = (long long)B * cin * (T / 4);
    int blocks = (int)std::min<long long>(ceil_div_ll(total, 256), (long long)num_sms() * 8);
    coupling_apply_kernel<4><<<blocks, 256, 0, st>>>(x, x_bstride, lst, z, z_bstride, neg_log_s, cin, T, inverse, total);
  } else {
    long long total = (long long)B * cin * T;
    int blocks = (int)std::min<long long>(ceil_div_ll(total, 256), (long long)num_sms() * 8);
    coupling_apply_kernel<1><<<blocks, 256, 0, st>>>(x, x_bstride, lst, z, z_bstride, neg_log_s, cin, T, inverse, total);
  }
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

int cmwg_coupling_apply_varlen(const float* x, long long x_bstride, const float* lst, float* z, long long z_bstride,
                               float* neg_log_s, int B, int cin, int T, const int* lengths_dev, int inverse, void* stream) {
  CMWG_REQUIRE(lengths_dev, "cmwg_coupling_apply_varlen: null lengths");
  if (B == 0 || T == 0 || cin == 0) return CMWG_OK;
  cudaStream_t st = (cudaStream_t)stream;
  bool vec = (T % 4 == 0) && (x_bstride % 4 == 0) && (z_bstride % 4 == 0) && (((uintptr_t)x & 15) == 0) &&
             (((uintptr_t)z & 15) == 0) && (((uintptr_t)lst & 15) == 0) && (((uintptr_t)neg_log_s & 15) == 0);
  if (vec) {
    long long total = (long long)B * cin * (T / 4);
    int blocks = (int)std::min<long long>(ceil_div_ll(total, 256), (long long)num_sms() * 8);
    coupling_apply_kernel<4><<<blocks, 256, 0, st>>>(x, x_bstride, lst, z, z_bstride, neg_log_s, cin, T, inverse, total,
                                                     lengths_dev);
  } else {
    long long total = (long long)B * cin * T;
    int blocks = (int)std::min<long long>(ceil_div_ll(total, 256), (long long)num_sms() * 8);
    coupling_apply_kernel<1><<<blocks, 256, 0, st>>>(x, x_bstride, lst, z, z_bstride, neg_log_s, cin, T, inverse, total,
                                                     lengths_dev);
  }
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

int cmwg_coupling_bwd(const float* out, long long out_bstride, const float* lst, const float* dout,
                      long long dout_bstride, const float* dls, long long dls_bstride, float* restored, float* dlst,
                      float* din, int B, int cin, int T, int inverse, void* stream) {
  if (B == 0 || T == 0 || cin == 0) return CMWG_OK;
  long long total = (long long)B * cin * T;
  int blocks = (int)std::min<long long>(ceil_div_ll(total, 256), (long long)num_sms() * 8);
  coupling_bwd_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(out, out_bstride, lst, dout, dout_bstride, dls,
                                                                dls_bstride, restored, dlst, din, cin, T, inverse,
                                                                total);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

int cmwg_squeeze(const float* x, float* out, int B, int T, int n_group, int inverse, void* stream) {
  CMWG_REQUIRE(n_group > 0 && T % n_group == 0, "cmwg_squeeze: T=%d not a multiple of n_group=%d", T, n_group);
  long long total = (long long)B * T;
  if (total == 0) return CMWG_OK;
  int blocks = (int)std::min<long long>(ceil_div_ll(total, 256), (long long)num_sms() * 8);
  squeeze_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(x, out, T / n_group, n_group, inverse, total);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

int cmwg_sum_per_batch(const float* a, long long a_bstride, int B, int N, float* out, int accumulate, float scale,
                       void* stream) {
  if (B == 0) return CMWG_OK;
  sum_per_batch_kernel<<<B, 1024, 0, (cudaStream_t)stream>>>(a, a_bstride, N, out, accumulate, scale);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

int cmwg_logdet_accumulate(const float* a, long long a_bstride, int B, int N, const float* prev, const float* log_det_w,
                           float* out, void* stream) {
  CMWG_REQUIRE(a && out, "cmwg_logdet_accumulate: null argument");
  if (B == 0) return CMWG_OK;
  logdet_accumulate_kernel<<<B, 1024, 0, (cudaStream_t)stream>>>(a, a_bstride, N, prev, log_det_w, out);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

int cmwg_logdet_accumulate_varlen(const float* a, long long a_bstride, int B, int C, int T, const int* lengths_dev,
                                  const float* prev, const float* log_det_w, float* out, void* stream) {
  CMWG_REQUIRE(a && out && lengths_dev, "cmwg_logdet_accumulate_varlen: null argument");
  if (B == 0) return CMWG_OK;
  logdet_accumulate_varlen_kernel<<<B, 1024, 0, (cudaStream_t)stream>>>(a, a_bstride, C, T, lengths_dev, prev, log_det_w, out);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

int cmwg_nll_loss(const float* z, const float* logdet, int B, int T, float sigma, int elementwise_mean, float* loss,
                  float* dz, void* workspace, void* stream) {
  CMWG_REQUIRE(B > 0 && T > 0, "cmwg_nll_loss: empty input");
  cudaStream_t st = (cudaStream_t)stream;
  float* rows = (float*)workspace;
  float inv_s2 = 1.f / (sigma * sigma);
  nll_rows_kernel<<<B, 1024, 0, st>>>(z, T, rows);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  nll_final_kernel<<<1, 32, 0, st>>>(rows, logdet, B, T, inv_s2, elementwise_mean, loss);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  if (dz) {
    float k = inv_s2 / (float)B / (elementwise_mean ? (float)T : 1.f);
    long long n = (long long)B * T;
    int blocks = (int)std::min<long long>(ceil_div_ll(n, 256), (long long)num_sms() * 8);
    scale_kernel<<<blocks, 256, 0, st>>>(z, dz, k, n);
    CMWG_COUNT_LAUNCH();
    CMWG_LAUNCH_CHECK();
  }
  return CMWG_OK;
}

}  // extern "C"
