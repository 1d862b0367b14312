// Exact fp32 GEMM engine on the CUDA cores (FFMA), used when TF32/bf16 rounding is not allowed
// (torch.backends.cudnn.allow_tf32 == False, i.e. the reference's tests and `train.py --no-tf32`)
// and for WN shapes the tcgen05 engine does not tile (channels not multiples of 64).
//
//   D[row][n] = sum_s sum_k A_s[row + shift_s][k] * W[n][koff_s + k]       (ff_gemm_kernel)
//   D[m][n]   = sum_t  A[t][m] * Bsrc[t + shift][n]                         (ff_wgrad_kernel)
// Rows are (batch, line, time): a slab is [B][H][T][C] with H = 1 for the 1-D WN of WaveGlow and
// H = squeezed height for WaveFlow's 2-D WN; a tap shifts time AND line, both zero padded.
//
// 128x128 CTA tile, BK = 16, 256 threads, 8x8 register tile per thread (split 4+4 so that the two
// column groups a thread owns are 64 apart: the gate epilogue needs exactly that pairing),
// register-staged double buffering.
#pragma once
#include "common.cuh"
#include "wn_layout.cuh"

namespace cmwg {

constexpr int FF_BM = 128, FF_BN = 128, FF_BK = 16, FF_THREADS = 256, FF_LD = 132;

struct GemmSeg {
  const void* a;  // slab [B*T][lda]
  int lda;
  int K;          // valid channels of this segment
  int shift;      // row (time) shift applied to the A operand
  int koff;       // column offset of this segment inside the weight matrix
  int shift_h;    // line (height) shift applied to the A operand (2-D WN)
  int bcast_h;    // the operand has no line dimension ([B][T][C], e.g. the conditioning): same rows for every line
};

struct GemmDesc {
  GemmSeg seg[MAX_SEG];
  int nseg;
  const void* w;  // [N][ldw] packed weights (operand type)
  int ldw;
  int N;          // valid output columns
  int n_rows_w;   // rows physically present in w (>= N, used for the TMA map)
  int B, T;
  int H;          // lines per batch item (0 or 1: plain [B][T] slabs)
  int h0, nh;     // line window: only lines [h0, h0 + nh) of every batch item are computed (nh = 0: all H lines);
                  // taps still read any line of the slab (row-recurrent inverse of the 2-D WN)
  int bn;         // N tile (tc engine)
  int is_fp16;
  int tag;        // CMWG_KCLASS_* for the profiler
  const int* row_len;  // nullptr, or per-item lengths (1-D WN): the epilogue writes 0 at rows t >= row_len[b] (tc engine)
};

struct FfGemmParams {
  GemmSeg seg[MAX_SEG];
  int nseg;
  const float* w;
  int ldw, N, B, T, H, tiles_per_batch;  // tiles_per_batch: tiles per LINE
  int h0, nh;                            // line window
};

__device__ __forceinline__ void ff_mma_tile(const float (*As)[FF_LD], const float (*Bs)[FF_LD], int tx, int ty,
                                            float (&acc)[8][8]) {
#pragma unroll
  for (int k = 0; k < FF_BK; ++k) {
    float4 a0 = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
    float4 a1 = *reinterpret_cast<const float4*>(&As[k][64 + ty * 4]);
    float4 b0 = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
    float4 b1 = *reinterpret_cast<const float4*>(&Bs[k][64 + tx * 4]);
    float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
    float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
  }
}

template <class Epi, bool PAIRED>
__global__ void __launch_bounds__(FF_THREADS) ff_gemm_kernel(const FfGemmParams p, const Epi epi) {
  __shared__ __align__(16) float As[2][FF_BK][FF_LD];
  __shared__ __align__(16) float Bs[2][FF_BK][FF_LD];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int wl = blockIdx.x / p.tiles_per_batch;  // line inside the window
  const int b = wl / p.nh, h = p.h0 + (wl - b * p.nh);
  const int line = b * p.H + h;
  const int t0 = (blockIdx.x % p.tiles_per_batch) * FF_BM;
  const int n0 = blockIdx.y * FF_BN;
  const int lr = tid >> 2;         // 0..63 : row inside the half tile
  const int kq = (tid & 3) * 4;    // k offset of this thread's float4

  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  // flattened (segment, k-block) iteration
  int total_kb = 0;
  for (int s = 0; s < p.nseg; ++s) total_kb += (p.seg[s].K + FF_BK - 1) / FF_BK;

  float4 ra[2], rb[2];
  auto fetch = [&](int s, int kb) {
    const GemmSeg& sg = p.seg[s];
    const float* ap = reinterpret_cast<const float*>(sg.a);
    int k = kb * FF_BK + kq;
    const int ha = h + sg.shift_h;
    const bool hok = sg.bcast_h || (ha >= 0 && ha < p.H);
    const long long line_a = sg.bcast_h ? (long long)b : (long long)b * p.H + ha;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      int t = t0 + lr + 64 * i + sg.shift;
      bool ok = hok && (t >= 0) && (t < p.T) && (k < sg.K);
      ra[i] = ok ? *reinterpret_cast<const float4*>(ap + (line_a * p.T + t) * sg.lda + k)
                 : make_float4(0.f, 0.f, 0.f, 0.f);
      int n = n0 + lr + 64 * i;
      bool okb = (n < p.N) && (k < sg.K);
      rb[i] = okb ? *reinterpret_cast<const float4*>(p.w + (long long)n * p.ldw + sg.koff + k)
                  : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto stash = [&](int buf) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      int r = lr + 64 * i;
      As[buf][kq + 0][r] = ra[i].x; As[buf][kq + 1][r] = ra[i].y;
      As[buf][kq + 2][r] = ra[i].z; As[buf][kq + 3][r] = ra[i].w;
      Bs[buf][kq + 0][r] = rb[i].x; Bs[buf][kq + 1][r] = rb[i].y;
      Bs[buf][kq + 2][r] = rb[i].z; Bs[buf][kq + 3][r] = rb[i].w;
    }
  };

  int s = 0, kb = 0;
  auto advance = [&]() {
    ++kb;
    if (kb * FF_BK >= p.seg[s].K) { kb = 0; ++s; }
  };
  fetch(s, kb);
  stash(0);
  __syncthreads();
  for (int it = 0; it < total_kb; ++it) {
    int cur = it & 1;
    advance();
    bool more = (it + 1) < total_kb;
    if (more) fetch(s, kb);
    ff_mma_tile(As[cur], Bs[cur], tx, ty, acc);
    if (more) stash(cur ^ 1);
    __syncthreads();
  }

#pragma unroll
  for (int ri = 0; ri < 8; ++ri) {
    int rl = (ri < 4) ? (ty * 4 + ri) : (64 + ty * 4 + ri - 4);
    int t = t0 + rl;
    if (t >= p.T) continue;
    long long row = (long long)line * p.T + t;
    float lo[4] = {acc[ri][0], acc[ri][1], acc[ri][2], acc[ri][3]};
    float hi[4] = {acc[ri][4], acc[ri][5], acc[ri][6], acc[ri][7]};
    if constexpr (PAIRED) {
      epi.template pair<4>(row, blockIdx.y * 64 + tx * 4, lo, hi);
    } else {
      int c0 = n0 + tx * 4, c1 = n0 + 64 + tx * 4;
      if (c0 < p.N) epi.template op<4>(row, c0, lo);
      if (c1 < p.N) epi.template op<4>(row, c1, hi);
    }
  }
}

template <class Epi, bool PAIRED>
int ff_gemm_launch(const GemmDesc& d, const Epi& epi, cudaStream_t st) {
  FfGemmParams p;
  for (int s = 0; s < d.nseg; ++s) {
    p.seg[s] = d.seg[s];
    CMWG_REQUIRE(d.seg[s].K % 4 == 0 && d.seg[s].lda % 4 == 0, "ff_gemm: segment K/lda must be multiples of 4");
  }
  p.nseg = d.nseg;
  p.w = reinterpret_cast<const float*>(d.w);
  p.ldw = d.ldw; p.N = d.N; p.B = d.B; p.T = d.T; p.H = d.H > 0 ? d.H : 1;
  p.tiles_per_batch = ceil_div(d.T, FF_BM);
  p.h0 = d.nh > 0 ? d.h0 : 0;
  p.nh = d.nh > 0 ? d.nh : p.H;
  CMWG_REQUIRE(p.h0 >= 0 && p.h0 + p.nh <= p.H, "gemm: line window [%d, %d) outside [0, %d)", p.h0, p.h0 + p.nh, p.H);
  dim3 grid(d.B * p.nh * p.tiles_per_batch, ceil_div(d.N, FF_BN));
  if (grid.x == 0 || grid.y == 0) return CMWG_OK;
  ProfScope prof(st, d.tag);
  ff_gemm_kernel<Epi, PAIRED><<<grid, FF_THREADS, 0, st>>>(p, epi);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

// ---- weight gradient: both operands MN-major (channel contiguous), K = time ---------------------
struct WgradProblem {
  const void* a; int lda; int a_c0; int M;   // A[t][a_c0 + m]
  const void* b; int ldb; int b_c0; int N;   // Bsrc[t + shift][b_c0 + n]
  int shift;
  int shift_h;                               // line shift of the B operand (2-D WN)
  int bcast_h;                               // B operand has no line dimension ([B][T][C])
  float* partial;                            // [splits][M][N]
};

struct FfWgradParams {
  WgradProblem pr;
  int B, T, H, Lc, chunks_per_batch, n_tiles_n;  // chunks_per_batch: chunks per LINE
};

static __global__ void __launch_bounds__(FF_THREADS) ff_wgrad_kernel(const FfWgradParams p) {
  __shared__ __align__(16) float As[2][FF_BK][FF_LD];
  __shared__ __align__(16) float Bs[2][FF_BK][FF_LD];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int m0 = (blockIdx.x / p.n_tiles_n) * FF_BM;
  const int n0 = (blockIdx.x % p.n_tiles_n) * FF_BN;
  const int split = blockIdx.y;
  const int line = split / p.chunks_per_batch;
  const int b = line / p.H, h = line - b * p.H;
  const int hb = h + p.pr.shift_h;
  const bool hok = p.pr.bcast_h || (hb >= 0 && hb < p.H);
  const long long line_b = p.pr.bcast_h ? (long long)b : (long long)b * p.H + hb;
  const int tc0 = (split % p.chunks_per_batch) * p.Lc;
  const int tlen = min(p.Lc, p.T - tc0);
  const float* A = reinterpret_cast<const float*>(p.pr.a);
  const float* Bm = reinterpret_cast<const float*>(p.pr.b);
  const int lk = tid >> 5;        // 0..7 (+8)
  const int c4 = (tid & 31) * 4;  // channel offset

  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  float4 ra[2], rb[2];
  auto fetch = [&](int kb) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      int k = kb * FF_BK + lk + 8 * i;
      int t = tc0 + k;
      bool oka = (k < tlen) && (m0 + c4 < p.pr.M);
      ra[i] = oka ? *reinterpret_cast<const float4*>(A + ((long long)line * p.T + t) * p.pr.lda + p.pr.a_c0 + m0 + c4)
                  : make_float4(0.f, 0.f, 0.f, 0.f);
      int tb = t + p.pr.shift;
      bool okb = hok && (k < tlen) && (tb >= 0) && (tb < p.T) && (n0 + c4 < p.pr.N);
      rb[i] = okb ? *reinterpret_cast<const float4*>(Bm + (line_b * p.T + tb) * p.pr.ldb + p.pr.b_c0 + n0 + c4)
                  : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto stash = [&](int buf) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      *reinterpret_cast<float4*>(&As[buf][lk + 8 * i][c4]) = ra[i];
      *reinterpret_cast<float4*>(&Bs[buf][lk + 8 * i][c4]) = rb[i];
    }
  };
  int nkb = (tlen + FF_BK - 1) / FF_BK;
  fetch(0);
  stash(0);
  __syncthreads();
  for (int it = 0; it < nkb; ++it) {
    int cur = it & 1;
    bool more = (it + 1) < nkb;
    if (more) fetch(it + 1);
    ff_mma_tile(As[cur], Bs[cur], tx, ty, acc);
    if (more) stash(cur ^ 1);
    __syncthreads();
  }
  float* out = p.pr.partial + (long long)split * p.pr.M * p.pr.N;
#pragma unroll
  for (int ri = 0; ri < 8; ++ri) {
    int m = m0 + ((ri < 4) ? (ty * 4 + ri) : (64 + ty * 4 + ri - 4));
    if (m >= p.pr.M) continue;
    int c0 = n0 + tx * 4, c1 = n0 + 64 + tx * 4;
    if (c0 < p.pr.N)
      *reinterpret_cast<float4*>(out + (long long)m * p.pr.N + c0) =
          make_float4(acc[ri][0], acc[ri][1], acc[ri][2], acc[ri][3]);
    if (c1 < p.pr.N)
      *reinterpret_cast<float4*>(out + (long long)m * p.pr.N + c1) =
          make_float4(acc[ri][4], acc[ri][5], acc[ri][6], acc[ri][7]);
  }
}

inline int ff_wgrad_launch(const WgradProblem& pr, int B, int H, int T, int Lc, cudaStream_t st) {
  CMWG_REQUIRE(pr.M % 4 == 0 && pr.N % 4 == 0 && pr.lda % 4 == 0 && pr.ldb % 4 == 0 && pr.a_c0 % 4 == 0 &&
                   pr.b_c0 % 4 == 0,
               "ff_wgrad: dims must be multiples of 4");
  FfWgradParams p;
  p.pr = pr; p.B = B; p.T = T; p.H = H > 0 ? H : 1; p.Lc = Lc;
  p.chunks_per_batch = ceil_div(T, Lc);
  p.n_tiles_n = ceil_div(pr.N, FF_BN);
  dim3 grid(ceil_div(pr.M, FF_BM) * p.n_tiles_n, B * p.H * p.chunks_per_batch);
  if (grid.x == 0 || grid.y == 0) return CMWG_OK;
  ProfScope prof(st, CMWG_KCLASS_WGRAD);
  ff_wgrad_kernel<<<grid, FF_THREADS, 0, st>>>(p);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

}  // namespace cmwg
