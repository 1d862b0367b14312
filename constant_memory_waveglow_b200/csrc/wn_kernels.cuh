// CUDA-core kernels around the WN GEMMs: weight norm (forward / backward), operand packing,
// conditioning layout change, the tiny-K `start` conv and tiny-N `end` conv (forward / backward),
// fixed-order reductions of block partials.
#pragma once
#include "common.cuh"
#include "epilogues.cuh"
#include "wn_layout.cuh"

namespace cmwg {

constexpr int ROWS_PER_BLOCK = 32;  // start/end conv kernels: rows (time steps) per CTA

// ------------------------------------------------------------------------------------------------
// deterministic block reduction (blockDim.x = 128)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float block_sum_128(float v, float* red /*[4]*/) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = red[0] + red[1] + red[2] + red[3];
  __syncthreads();
  return r;
}

// ------------------------------------------------------------------------------------------------
// weight norm forward for ALL convs of one WN in one launch  (utils.py:14-16 -> torch weight_norm)
// ------------------------------------------------------------------------------------------------
struct WeffEntry {
  const float* g;  // nullptr: no weight norm (w = v)
  const float* v;
  float* w;        // effective weight out, same layout as v
  float* inv_norm; // [O] or nullptr
  int O, L;        // out channels, elements per out channel
  int row_begin;   // prefix sum of O
};
struct WeffTable {
  WeffEntry e[2 * CMWG_MAX_DEPTH + 3];
  int n;
};

static __global__ void __launch_bounds__(128) weight_eff_kernel(const WeffTable tb) {
  __shared__ float red[4];
  int row = blockIdx.x;
  int ci = 0;
  while (ci + 1 < tb.n && row >= tb.e[ci + 1].row_begin) ++ci;
  const WeffEntry& e = tb.e[ci];
  int o = row - e.row_begin;
  const float* v = e.v + (long long)o * e.L;
  float* w = e.w + (long long)o * e.L;
  if (e.g == nullptr) {
    for (int l = threadIdx.x; l < e.L; l += 128) w[l] = v[l];
    return;
  }
  float ss = 0.f;
  for (int l = threadIdx.x; l < e.L; l += 128) ss = fmaf(v[l], v[l], ss);
  ss = block_sum_128(ss, red);
  float norm = sqrtf(ss);
  float scale = e.g[o] / norm;
  for (int l = threadIdx.x; l < e.L; l += 128) w[l] = v[l] * scale;
  if (threadIdx.x == 0 && e.inv_norm) e.inv_norm[o] = 1.f / norm;
}

// weight norm backward for ALL convs of one WN in one launch: (dw_eff, v, g, 1/||v||) -> (dg, dv);
// without weight norm dv = dw_eff.  One CTA per output channel.
// A row of the effective-weight gradient may also be GATHERED from the full-K tiles the batched weight-gradient launch
// leaves behind (one tile per tap / per W_o row block, see wn_pipeline.cu): source j covers rows [row0, row0 + M) of the
// conv and writes tile element (m, n) to position col0 + n * sn of row row0 + m.  That folds the split-K "reduce" pass (a
// pure re-layout when there is a single split) into this kernel.
struct WnBwdSrc {
  const float* tile;   // [M][ld] fp32
  int M, ld, n_valid;  // rows, row pitch, valid columns
  int row0, col0, sn;  // destination row offset, column offset, column stride
};
constexpr int WN_BWD_MAX_SRC = 8;   // radix <= 7 taps of W, or the two row blocks of W_o
struct WnBwdEntry {
  const float* dw;        // effective-weight gradient, natural layout [O][L] (used when nsrc == 0)
  const float* v;
  const float* g;         // nullptr: no weight norm
  const float* inv_norm;  // [O]
  float* dg;              // nullptr: not wanted
  float* dv;
  int O, L;
  int row_begin;          // prefix sum of O
  int nsrc;
  WnBwdSrc src[WN_BWD_MAX_SRC];
};
struct WnBwdTable {
  WnBwdEntry e[3 * CMWG_MAX_DEPTH + 2];
  int n;
  const float* gscale;    // nullptr, or the gradient-scale triple: gathered tiles are multiplied by gscale[2] = 1 / S
};

constexpr int WN_BWD_MAX_L = 7 * 256;   // longest conv row gathered through shared memory (radix 7 x 256 channels)

static __global__ void __launch_bounds__(128) weight_norm_bwd_kernel(const __grid_constant__ WnBwdTable tb) {
  __shared__ float red[4];
  __shared__ __align__(16) float rowbuf[WN_BWD_MAX_L];
  int row = blockIdx.x;
  int ci = 0;
  while (ci + 1 < tb.n && row >= tb.e[ci + 1].row_begin) ++ci;
  const WnBwdEntry& e = tb.e[ci];
  const int o = row - e.row_begin, L = e.L;
  const float* dwo = e.dw + (long long)o * L;
  if (e.nsrc > 0) {
    const float inv_scale = tb.gscale ? tb.gscale[2] : 1.f;
    for (int j = 0; j < e.nsrc; ++j) {
      const WnBwdSrc& sj = e.src[j];
      const int m = o - sj.row0;
      if (m < 0 || m >= sj.M) continue;
      const float* t = sj.tile + (long long)m * sj.ld;
      for (int n = threadIdx.x; n < sj.n_valid; n += 128) rowbuf[sj.col0 + n * sj.sn] = t[n] * inv_scale;
    }
    __syncthreads();
    dwo = rowbuf;
  }
  if (e.g == nullptr) {
    if (e.dv)
      for (int l = threadIdx.x; l < L; l += 128) e.dv[(long long)o * L + l] = dwo[l];
    return;
  }
  const float* vo = e.v + (long long)o * L;
  float* dvo = e.dv ? e.dv + (long long)o * L : nullptr;
  // rows of whole, 16-byte aligned float4 (every conv of the shipped configs but the start conv): a quarter of the instructions
  const bool vec = (L & 3) == 0 && (((uintptr_t)vo | (uintptr_t)dwo | (uintptr_t)dvo) & 15) == 0;
  float dot = 0.f;
  if (vec) {
    for (int l = threadIdx.x * 4; l < L; l += 512) {
      const float4 a = *reinterpret_cast<const float4*>(dwo + l), b = *reinterpret_cast<const float4*>(vo + l);
      dot = fmaf(a.x, b.x, dot); dot = fmaf(a.y, b.y, dot); dot = fmaf(a.z, b.z, dot); dot = fmaf(a.w, b.w, dot);
    }
  } else {
    for (int l = threadIdx.x; l < L; l += 128) dot = fmaf(dwo[l], vo[l], dot);
  }
  dot = block_sum_128(dot, red);
  float inv = e.inv_norm[o];
  if (threadIdx.x == 0 && e.dg) e.dg[o] = dot * inv;
  if (dvo) {
    float gs = e.g[o] * inv;
    float k = dot * inv * inv;
    if (vec) {
      for (int l = threadIdx.x * 4; l < L; l += 512) {
        const float4 a = *reinterpret_cast<const float4*>(dwo + l), b = *reinterpret_cast<const float4*>(vo + l);
        *reinterpret_cast<float4*>(dvo + l) =
            make_float4(gs * (a.x - b.x * k), gs * (a.y - b.y * k), gs * (a.z - b.z * k), gs * (a.w - b.w * k));
      }
    } else {
      for (int l = threadIdx.x; l < L; l += 128) dvo[l] = gs * (dwo[l] - vo[l] * k);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// operand packing: one launch packs the five GEMM matrices of every layer
// ------------------------------------------------------------------------------------------------
struct PackParams {
  WnDims d;
  const float* wV;
  const float* wW[CMWG_MAX_DEPTH];
  const float* wWo[CMWG_MAX_DEPTH];
  void* PA[CMWG_MAX_DEPTH];
  void* PB[CMWG_MAX_DEPTH];
  void* Q1[CMWG_MAX_DEPTH];
  void* Q2[CMWG_MAX_DEPTH];
  void* QV;  // shared [auxp][ldQV]
  void* PS;  // [Cs][ldPS] (tc)
  int is_fp16;
};

template <typename OpT>
static __global__ void __launch_bounds__(256) pack_operands_kernel(const PackParams p) {
  const WnDims& d = p.d;
  const int i = blockIdx.y;     // layer
  const int kind = blockIdx.z;  // 0 PA, 1 PB, 2 Q1, 3 Q2, 4 QV, 5 PS
  const int nb = d.nb(i), k1 = d.k1(i), cr_eff = d.cr_eff(i);
  long long size;
  switch (kind) {
    case 0: size = (long long)d.npadA * d.KA; break;
    case 1: size = (long long)nb * d.ldPB; break;
    case 2: size = (long long)d.Cd * k1; break;
    case 3: size = (long long)d.Cr * d.ldQ2; break;
    case 4: size = (long long)d.auxp * d.Cd2p; break;
    default: size = d.tc ? (long long)d.Cs * d.Cdp : 0; break;
  }
  const float* wW = p.wW[i];
  const float* wWo = p.wWo[i];
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < size;
       idx += (long long)gridDim.x * blockDim.x) {
    float val = 0.f;
    OpT* dst;
    long long didx = idx;  // destination element index (differs from idx for the K-concatenated matrices)
    if (kind == 0) {
      int n = (int)(idx / d.KA), k = (int)(idx % d.KA);
      int tile = n / d.bn_gate, r = n % d.bn_gate;
      int half = r / d.G, ch = tile * d.G + (r % d.G);
      if (ch < d.Cd) {
        int oc = half * d.Cd + ch;
        if (k < d.R * d.Crp) {
          int tap = k / d.Crp, ic = k % d.Crp;
          if (ic < d.Cr) val = wW[((long long)oc * d.Cr + ic) * d.R + tap];
        } else {
          int kk = k - d.R * d.Crp;
          if (kk < d.aux) val = p.wV[((long long)i * 2 * d.Cd + oc) * d.aux + kk];
        }
      }
      dst = reinterpret_cast<OpT*>(p.PA[i]);
    } else if (kind == 1) {
      int n = (int)(idx / d.ldPB), k = (int)(idx % d.ldPB);
      if (k < d.Cd) val = wWo[(long long)n * d.Cd + k];
      dst = reinterpret_cast<OpT*>(p.PB[i]);
    } else if (kind == 2) {
      int n = (int)(idx / k1), k = (int)(idx % k1);
      int ro = -1;
      if (cr_eff > 0) {
        if (k < d.Crp) { if (k < d.Cr) ro = k; }
        else { int kk = k - d.Crp; if (kk < d.Cs) ro = d.Cr + kk; }
      } else {
        if (k < d.Cs) ro = k;
      }
      if (ro >= 0) val = wWo[(long long)ro * d.Cd + n];
      dst = reinterpret_cast<OpT*>(p.Q1[i]);
    } else if (kind == 3) {
      int ld = d.ldQ2;
      int n = (int)(idx / ld), k = (int)(idx % ld);
      int tap = k / d.Cd2p, oc = k % d.Cd2p;
      if (oc < 2 * d.Cd) val = wW[((long long)oc * d.Cr + n) * d.R + tap];
      dst = reinterpret_cast<OpT*>(p.Q2[i]);
    } else if (kind == 4) {
      int n = (int)(idx / d.Cd2p), k = (int)(idx % d.Cd2p);
      if (n < d.aux && k < 2 * d.Cd) val = p.wV[((long long)i * 2 * d.Cd + k) * d.aux + n];
      dst = reinterpret_cast<OpT*>(p.QV);
      didx = (long long)n * d.ldQV + (long long)i * d.Cd2p + k;
    } else {
      int n = (int)(idx / d.Cdp), k = (int)(idx % d.Cdp);
      if (k < d.Cd) val = wWo[((long long)cr_eff + n) * d.Cd + k];
      dst = reinterpret_cast<OpT*>(p.PS);
      didx = (long long)n * d.ldPS + (long long)i * d.Cdp + k;
    }
    OpTraits<OpT>::store(dst + didx, val, p.is_fp16);
  }
}

// 16-bit operands: the same matrices, 8 or 16 destination-contiguous elements per thread (16 / 32-byte stores) with the work
// items ordered so that a warp's READS are contiguous too -- for the transposing matrices (Q1, Q2, QV) the lanes walk the
// source's fast axis and every lane writes its own full 32-byte sector.  (One element per thread took 56 us per WN at the LJ
// config, every training step, for 20 MB of output.)  Bit-identical to pack_operands_kernel<uint16_t>.
__device__ __forceinline__ void pack_store8(uint16_t* dst, const float (&v)[8], int f16) {
  *reinterpret_cast<uint4*>(dst) =
      make_uint4(pack2(v[0], v[1], f16), pack2(v[2], v[3], f16), pack2(v[4], v[5], f16), pack2(v[6], v[7], f16));
}
static __global__ void __launch_bounds__(256) pack_operands16_kernel(const PackParams p) {
  const WnDims& d = p.d;
  const int i = blockIdx.y;     // layer
  const int kind = blockIdx.z;  // 0 PA, 1 PB, 2 Q1, 3 Q2, 4 QV, 5 PS
  const int nb = d.nb(i), k1 = d.k1(i), cr_eff = d.cr_eff(i), f16 = p.is_fp16;
  const float* __restrict__ wW = p.wW[i];
  const float* __restrict__ wWo = p.wWo[i];
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long w0 = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (kind == 0) {
    uint16_t* dst = reinterpret_cast<uint16_t*>(p.PA[i]);
    const int wa = d.Crp / 8, per_row = wa + d.auxp / 8;
    for (long long w = w0; w < (long long)d.npadA * per_row; w += stride) {
      const int n = (int)(w / per_row), r = (int)(w % per_row);
      const int tile = n / d.bn_gate, rr = n % d.bn_gate;
      const int half = rr / d.G, ch = tile * d.G + (rr % d.G);
      const bool live = ch < d.Cd;
      const int oc = half * d.Cd + ch;
      float v[8];
      if (r < wa) {          // the taps of 8 consecutive input channels: 8 * R consecutive source floats
        const int ic0 = r * 8;
        for (int tap = 0; tap < d.R; ++tap) {
#pragma unroll
          for (int j = 0; j < 8; ++j)
            v[j] = (live && ic0 + j < d.Cr) ? wW[((long long)oc * d.Cr + ic0 + j) * d.R + tap] : 0.f;
          pack_store8(dst + (long long)n * d.KA + tap * d.Crp + ic0, v, f16);
        }
      } else {               // conditioning columns
        const int kk0 = (r - wa) * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j)
          v[j] = (live && kk0 + j < d.aux) ? p.wV[((long long)i * 2 * d.Cd + oc) * d.aux + kk0 + j] : 0.f;
        pack_store8(dst + (long long)n * d.KA + d.R * d.Crp + kk0, v, f16);
      }
    }
  } else if (kind == 1 || kind == 5) {
    if (kind == 5 && !d.tc) return;
    const int rows = kind == 1 ? nb : d.Cs, ld = kind == 1 ? d.ldPB : d.Cdp, per_row = ld / 8;
    const int row_off = kind == 1 ? 0 : cr_eff;
    uint16_t* dst = reinterpret_cast<uint16_t*>(kind == 1 ? p.PB[i] : p.PS);
    for (long long w = w0; w < (long long)rows * per_row; w += stride) {
      const int n = (int)(w / per_row), k0 = (int)(w % per_row) * 8;
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = (k0 + j < d.Cd) ? wWo[((long long)row_off + n) * d.Cd + k0 + j] : 0.f;
      pack_store8(dst + (kind == 1 ? (long long)n * d.ldPB + k0 : (long long)n * d.ldPS + (long long)i * d.Cdp + k0), v, f16);
    }
  } else if (kind == 2) {    // Q1 = W_o^T: lanes walk n (the source's fast axis), 16 k per thread
    uint16_t* dst = reinterpret_cast<uint16_t*>(p.Q1[i]);
    for (long long w = w0; w < (long long)d.Cd * (k1 / 16); w += stride) {
      const int n = (int)(w % d.Cd), k0 = (int)(w / d.Cd) * 16;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int k = k0 + 8 * h + j;
          int ro = -1;
          if (cr_eff > 0) {
            if (k < d.Crp) { if (k < d.Cr) ro = k; }
            else { const int kk = k - d.Crp; if (kk < d.Cs) ro = d.Cr + kk; }
          } else {
            if (k < d.Cs) ro = k;
          }
          v[j] = ro >= 0 ? wWo[(long long)ro * d.Cd + n] : 0.f;
        }
        pack_store8(dst + (long long)n * k1 + k0 + 8 * h, v, f16);
      }
    }
  } else if (kind == 3) {    // Q2 = W^T per tap: lanes walk n, 16 output channels x R taps per thread
    uint16_t* dst = reinterpret_cast<uint16_t*>(p.Q2[i]);
    for (long long w = w0; w < (long long)d.Cr * (d.Cd2p / 16); w += stride) {
      const int n = (int)(w % d.Cr), oc0 = (int)(w / d.Cr) * 16;
      for (int tap = 0; tap < d.R; ++tap) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float v[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int oc = oc0 + 8 * h + j;
            v[j] = oc < 2 * d.Cd ? wW[((long long)oc * d.Cr + n) * d.R + tap] : 0.f;
          }
          pack_store8(dst + (long long)n * d.ldQ2 + tap * d.Cd2p + oc0 + 8 * h, v, f16);
        }
      }
    }
  } else {                   // QV = V^T, K-concatenated over layers: lanes walk n
    uint16_t* dst = reinterpret_cast<uint16_t*>(p.QV);
    for (long long w = w0; w < (long long)d.auxp * (d.Cd2p / 16); w += stride) {
      const int n = (int)(w % d.auxp), k0 = (int)(w / d.auxp) * 16;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int k = k0 + 8 * h + j;
          v[j] = (n < d.aux && k < 2 * d.Cd) ? p.wV[((long long)i * 2 * d.Cd + k) * d.aux + n] : 0.f;
        }
        pack_store8(dst + (long long)n * d.ldQV + (long long)i * d.Cd2p + k0 + 8 * h, v, f16);
      }
    }
  }
}

// Layer 0 with the start conv folded in (wn_layout.cuh: PA0f / PB0f).  Column aux + tap * cin + c of the conditioning slab
// holds x_a[c] at the tap's time offset, so
//   PA0f[n][aux + tap * cin + c] = sum_ic W_0[oc(n)][ic][tap] * W_start[ic][c]      (gate rows in PA's interleaved order)
//   PB0f[n][Cdp + j]             = W_start[n][c]  where column (auxp - kb) + j is the centre tap's channel c
// and everything else is PA's conditioning block / PB's W_o block / zero.
struct Fold0Params {
  WnDims d;
  const float* wV;      // [depth * 2Cd][aux]
  const float* wW0;     // [2Cd][Cr][R]
  const float* wWo0;    // [nb(0)][Cd]
  const float* wStart;  // [Cr][cin]
  uint16_t* PA0f;
  uint16_t* PB0f;
  int is_fp16;
};
// PA0f[n][aux + tap * cin + c] = sum_ic W_0[oc(n)][ic][tap] * W_start[ic][c]: one warp per element, lanes stride the input
// channels (fixed shuffle order: deterministic)
__device__ __forceinline__ void pack_fold0_dot(const Fold0Params& p, int block) {
  const WnDims& d = p.d;
  const int per = d.R * d.cin, lane = threadIdx.x & 31;
  const long long wid = (block * 256ll + threadIdx.x) >> 5;
  if (wid >= (long long)d.npadA * per) return;
  const int n = (int)(wid / per), j = (int)(wid % per), tap = j / d.cin, c = j % d.cin;
  const int tile = n / d.bn_gate, r = n % d.bn_gate;
  const int half = r / d.G, ch = tile * d.G + (r % d.G);
  float val = 0.f;
  if (ch < d.Cd) {
    const float* w = p.wW0 + (long long)(half * d.Cd + ch) * d.Cr * d.R + tap;
    for (int ic = lane; ic < d.Cr; ic += 32) val = fmaf(w[(long long)ic * d.R], p.wStart[ic * d.cin + c], val);
    val = warp_sum(val);
  }
  if (lane == 0) p.PA0f[(long long)n * d.auxp + d.aux + j] = f32_to_op16(val, p.is_fp16);
}

static __global__ void __launch_bounds__(256) pack_fold0_kernel(const Fold0Params p) {
  const WnDims& d = p.d;
  const long long nA = (long long)d.npadA * d.auxp, ldB = d.Cdp + d.kb, nB = (long long)d.Cr * ldB;
  // blocks [0, nb_elem): one element per thread; blocks behind them: the folded columns, one warp per element
  const int nb_elem = (int)((nA + nB + 255) / 256);
  if ((int)blockIdx.x >= nb_elem) {
    pack_fold0_dot(p, blockIdx.x - nb_elem);
    return;
  }
  for (long long idx = blockIdx.x * 256ll + threadIdx.x; idx < nA + nB; idx += (long long)nb_elem * 256) {
    float val = 0.f;
    if (idx < nA) {
      const int n = (int)(idx / d.auxp), k = (int)(idx % d.auxp);
      const int tile = n / d.bn_gate, r = n % d.bn_gate;
      const int half = r / d.G, ch = tile * d.G + (r % d.G);
      if (ch < d.Cd) {
        const int oc = half * d.Cd + ch;
        if (k < d.aux) {
          val = p.wV[(long long)oc * d.aux + k];
        }   // the folded columns [aux, aux + R * cin) are 256-term dot products: pack_fold0_dot_kernel, one warp each
      }
      if (k < d.aux || k >= d.aux + d.R * d.cin) p.PA0f[idx] = f32_to_op16(val, p.is_fp16);
    } else {
      const long long j = idx - nA;
      const int n = (int)(j / ldB), k = (int)(j % ldB);
      if (k < d.Cd) {
        val = p.wWo0[(long long)n * d.Cd + k];
      } else if (k >= d.Cdp) {
        const int col = d.auxp - d.kb + (k - d.Cdp);               // column of the conditioning slab
        const int c = col - d.aux - ((d.R - 1) / 2) * d.cin;       // channel under the centre tap
        if (c >= 0 && c < d.cin) val = p.wStart[n * d.cin + c];
      }
      p.PB0f[j] = f32_to_op16(val, p.is_fp16);
    }
  }
}

// dgate weights with the `end` conv folded in (wn_layout.cuh: Q1f):  Q1f[i][n][k] = W_o,i[k][n] for k < Cr (layers with a
// residual half), and behind them one k-block whose first 2 in_channels columns hold
//   F_i[n][o] = sum_k W_o,i[cr_eff + k][n] * W_end[o][k]        (one warp per element, fixed shuffle order)
struct FoldEndParams {
  WnDims d;
  const float* wWo[CMWG_MAX_DEPTH];
  const float* wEnd;   // [2 cin][Cs]
  uint16_t* Q1f[CMWG_MAX_DEPTH];
  int is_fp16;
};
static __global__ void __launch_bounds__(256) pack_foldend_kernel(const FoldEndParams p) {
  const WnDims& d = p.d;
  const int i = blockIdx.y, cout = 2 * d.cin, cr_eff = d.cr_eff(i), ld = (i < d.depth - 1 ? d.Crp : 0) + d.kb;
  const int kres = ld - d.kb, f16 = p.is_fp16;
  const float* __restrict__ wWo = p.wWo[i];
  uint16_t* dst = p.Q1f[i];
  // blocks [0, nb_t): the transposed residual rows, lanes walk n (the source's fast axis), 16 k per thread (one 32-byte
  // sector); columns behind the residual rows are zero except the folded ones
  const int nb_t = (d.Cd * (ld / 16) + 255) / 256;
  if ((int)blockIdx.x < nb_t) {
    const int w = blockIdx.x * 256 + threadIdx.x;
    if (w >= d.Cd * (ld / 16)) return;
    const int n = w % d.Cd, k0 = (w / d.Cd) * 16;
    if (k0 >= kres && k0 < kres + 16) return;          // the k-group that holds the folded columns: written below
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int k = k0 + 8 * h + j;
        v[j] = (k < kres && k < d.Cr) ? wWo[(long long)k * d.Cd + n] : 0.f;
      }
      pack_store8(dst + (long long)n * ld + k0 + 8 * h, v, f16);
    }
    return;
  }
  // blocks behind them: F_i[n][o] for 32 consecutive n.  Thread (n, kg) sums its 32 skip rows for every o (coalesced
  // reads over n, W_end from shared memory), the 8 row groups fold in a fixed order.
  __shared__ float wend[16 * 32 * 8];     // [o][k within the group][kg]  (<= 16 outputs)
  __shared__ float part[8][16][33];
  const int nblk = blockIdx.x - nb_t;     // 32-wide n chunk
  const int nl = threadIdx.x & 31, kg = threadIdx.x >> 5;
  const int n = nblk * 32 + nl;
  const int per = d.Cs / 8;               // skip rows per group (Cs is a multiple of 64)
  float acc[16];
#pragma unroll
  for (int o = 0; o < 16; ++o) acc[o] = 0.f;
  for (int k0 = 0; k0 < per; k0 += 32) {
    __syncthreads();
    for (int idx = threadIdx.x; idx < cout * 32 * 8; idx += 256) {
      const int o = idx / 256, r = idx % 256, kk = r / 8, g = r % 8;
      const int k = g * per + k0 + kk;
      wend[idx] = (k0 + kk < per) ? p.wEnd[(long long)o * d.Cs + k] : 0.f;
    }
    __syncthreads();
    if (n < d.Cd) {
      for (int kk = 0; kk < 32 && k0 + kk < per; ++kk) {
        const float w = wWo[((long long)cr_eff + kg * per + k0 + kk) * d.Cd + n];
#pragma unroll
        for (int o = 0; o < 16; ++o)
          if (o < cout) acc[o] = fmaf(w, wend[(o * 32 + kk) * 8 + kg], acc[o]);
      }
    }
  }
#pragma unroll
  for (int o = 0; o < 16; ++o) part[kg][o][nl] = acc[o];
  __syncthreads();
  // 32 n x 16 columns of the folded k-group: thread (n, o) folds the 8 groups and the warp-wide store order is irrelevant
  for (int idx = threadIdx.x; idx < 32 * 16; idx += 256) {
    const int nn = idx & 31, o = idx >> 5;
    float sacc = 0.f;
    if (o < cout)
      for (int g = 0; g < 8; ++g) sacc += part[g][o][nn];
    if (nblk * 32 + nn < d.Cd) dst[(long long)(nblk * 32 + nn) * ld + kres + o] = f32_to_op16(sacc, f16);
  }
}

// S * d(log_s, t) as a [rows][kb] operand slab: the first 2 in_channels columns, zeros behind (folded `end` conv backward)
static __global__ void __launch_bounds__(256) dl_slab_kernel(const float* __restrict__ dlst, int cout, int T, long long rows,
                                                             int kb, uint16_t* __restrict__ dl, int is_fp16,
                                                             const float* __restrict__ gscale) {
  pdl_trigger();
  pdl_wait();
  const float sc = gscale ? gscale[1] : 1.f;
  const int groups = kb / 8;
  for (long long idx = blockIdx.x * 256ll + threadIdx.x; idx < rows * groups; idx += (long long)gridDim.x * 256) {
    // consecutive threads walk consecutive rows of one 8-column group: coalesced reads of dlst (B, cout, T)
    const long long row = idx % rows;
    const int gi = (int)(idx / rows);
    const int b = (int)(row / T), t = (int)(row - (long long)b * T);
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int o = gi * 8 + j;
      v[j] = o < cout ? dlst[((long long)b * cout + o) * T + t] * sc : 0.f;
    }
    pack_store8(dl + row * kb + gi * 8, v, is_fp16);
  }
}

// Weight gradients through the folded `end` conv.  The skip rows of every W_o and the `end` weight itself only ever see
// dskip = W_end^T d(log_s, t), so with  P_i[n][o] = sum_t g_i[t][n] * S d(log_s, t)[t][o]  (one small weight-gradient problem
// per layer, N = 2 in_channels instead of 256):
//   dW_o,i[cr_eff + k][n] = (1/S) sum_o W_end[o][k] P_i[n][o]
//   dW_end[o][k]          = (1/S) sum_i sum_n P_i[n][o] W_o,i[cr_eff + k][n]       (partials per layer, folded afterwards)
// neither the 256-channel dskip slab nor the saved fp32 skip sum is read.  grid (Cs / 32, depth), 256 threads.
struct FoldEndDwParams {
  const float* pred;                    // [depth][Cd][cout]: the P problems, split-K partials folded and 1 / S applied
                                        // (the reduce pass of the weight-gradient launch writes them)
  const float* wWo[CMWG_MAX_DEPTH];     // effective W_o, [nb(i)][Cd]
  float* dWo_skip[CMWG_MAX_DEPTH];      // [Cs][Cd] skip rows of the effective-weight gradient
  const float* wEnd;                    // [cout][Cs]
  float* dEnd_part;                     // [depth][cout][Cs] or nullptr
  int depth, Cd, Cs, Cr, cout;
};
constexpr int FOLDEND_DW_ROWS = 16;    // skip rows (k) per CTA
static __global__ void __launch_bounds__(256) foldend_dw_kernel(const FoldEndDwParams p) {
  __shared__ float Ps[256 * 16];                  // [n][o]   (Cd == 256, cout <= 16)
  __shared__ float Wt[FOLDEND_DW_ROWS][257];      // W_o,i skip rows of this block's k range, [k][n]
  const int i = blockIdx.y, kc = blockIdx.x * FOLDEND_DW_ROWS, cr_eff = i < p.depth - 1 ? p.Cr : 0;
  const float* __restrict__ pred = p.pred + (long long)i * p.Cd * p.cout;
#pragma unroll 4
  for (int idx = threadIdx.x; idx < p.Cd * 16; idx += 256) {
    const int n = idx >> 4, o = idx & 15;
    Ps[idx] = o < p.cout ? pred[n * p.cout + o] : 0.f;
  }
  for (int idx = threadIdx.x; idx < FOLDEND_DW_ROWS * p.Cd; idx += 256) {
    const int k = idx / p.Cd, n = idx - k * p.Cd;
    Wt[k][n] = p.wWo[i][((long long)cr_eff + kc + k) * p.Cd + n];
  }
  __syncthreads();
  // skip rows of dW_o,i: thread = n
  {
    const int n = threadIdx.x;
    float pr[16];
#pragma unroll
    for (int o = 0; o < 16; ++o) pr[o] = Ps[n * 16 + o];
    for (int k = 0; k < FOLDEND_DW_ROWS; ++k) {
      float a = 0.f;
#pragma unroll
      for (int o = 0; o < 16; ++o)
        if (o < p.cout) a = fmaf(p.wEnd[(long long)o * p.Cs + kc + k], pr[o], a);
      p.dWo_skip[i][((long long)kc + k) * p.Cd + n] = a;
    }
  }
  // this layer's share of dW_end[o][kc .. kc + 16): thread = (k, o), the n sum runs in a fixed order
  if (p.dEnd_part) {
    const int k = threadIdx.x >> 4, o = threadIdx.x & 15;
    float a = 0.f;
    for (int n = 0; n < p.Cd; ++n) a = fmaf(Ps[n * 16 + o], Wt[k][n], a);
    if (o < p.cout) p.dEnd_part[((long long)i * p.cout + o) * p.Cs + kc + k] = a;
  }
}

// taps of x_a into the padding columns of the conditioning slab: ycl[row][aux + tap * cin + c] = x[b][c][t + (tap - centre)]
// (zero outside [0, T), or [0, row_len[b]): the dilated conv's 'same' padding of h_0 = W_start x_a, which has no bias here)
static __global__ void __launch_bounds__(256) cond_aug_kernel(const float* __restrict__ x, long long x_bs, int cin, int R,
                                                              int B, int T, uint16_t* __restrict__ ycl, int aux, int auxp,
                                                              int is_fp16, const int* __restrict__ row_len) {
  pdl_trigger();
  pdl_wait();
  const long long rows = (long long)B * T;
  const int per = R * cin, ct = (R - 1) / 2;
  for (long long idx = blockIdx.x * 256ll + threadIdx.x; idx < rows * per; idx += (long long)gridDim.x * 256) {
    // consecutive threads walk consecutive time steps of one (tap, channel): coalesced reads
    const long long row = idx % rows;
    const int j = (int)(idx / rows), tap = j / cin, c = j % cin;
    const int b = (int)(row / T), t = (int)(row - (long long)b * T);
    const int ts = t + tap - ct;
    const int tv = row_len ? row_len[b] : T;   // per-item lengths: x_a is zero from the item's end on, as past T
    const float v = (ts >= 0 && ts < tv) ? x[b * x_bs + (long long)c * T + ts] : 0.f;
    ycl[row * auxp + aux + j] = f32_to_op16(v, is_fp16);
  }
}

// Weight gradient of layer 0's dilated conv through the fold.  With h_0 = W_start x_a never materialised,
//   dW_0[oc][ic][tap] = sum_t dpre_0[t][oc] h_0[t + shift_tap][ic] = sum_c D[oc][tap * cin + c] W_start[ic][c],
//   D[oc][tap * cin + c] = sum_t dpre_0[t][oc] x_a[c][t + shift_tap]
// and D is what the conditioning weight-gradient GEMM of layer 0 (dV_0 = dpre_0^T ycond) leaves in the columns of its tile
// that face the x_a taps in the conditioning slab: columns [aux, aux + R * cin).  One CTA per output channel.
static __global__ void __launch_bounds__(256) fold0_dw_kernel(const float* __restrict__ tile, int splits, int M, int N, int aux,
                                                              int cin, int R, int Cr, const float* __restrict__ wStart,
                                                              const float* __restrict__ gscale, float* __restrict__ dW) {
  __shared__ float Drow[64];
  const int oc = blockIdx.x, per = R * cin;
  if (threadIdx.x < per) {
    float sacc = 0.f;
    for (int j = 0; j < splits; ++j) sacc += tile[((long long)j * M + oc) * N + aux + threadIdx.x];   // fixed order
    Drow[threadIdx.x] = sacc * (gscale ? gscale[2] : 1.f);
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < Cr * R; idx += 256) {
    const int ic = idx / R, tap = idx - ic * R;
    float a = 0.f;
    for (int c = 0; c < cin; ++c) a = fmaf(Drow[tap * cin + c], wStart[ic * cin + c], a);
    dW[(long long)oc * Cr * R + idx] = a;
  }
}

struct BiasPackParams {
  WnDims d;
  const float* bV;
  const float* bStart;
  const float* bEnd;
  const float* bW[CMWG_MAX_DEPTH];
  const float* bWo[CMWG_MAX_DEPTH];
  float* biasA[CMWG_MAX_DEPTH];
  float* biasB[CMWG_MAX_DEPTH];
  float* biasStart;
  float* biasEnd;
  float* biasS;
};
static __global__ void __launch_bounds__(256) pack_bias_kernel(const BiasPackParams p) {
  const WnDims& d = p.d;
  int i = blockIdx.y;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < 2 * d.Cd; idx += gridDim.x * blockDim.x)
    p.biasA[i][idx] = p.bW[i][idx] + p.bV[i * 2 * d.Cd + idx];
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < d.nb(i); idx += gridDim.x * blockDim.x)
    p.biasB[i][idx] = p.bWo[i][idx];
  if (i == 0) {
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < d.Cr; idx += gridDim.x * blockDim.x)
      p.biasStart[idx] = p.bStart[idx];
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < 2 * d.cin; idx += gridDim.x * blockDim.x)
      p.biasEnd[idx] = p.bEnd[idx];
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < d.Cs; idx += gridDim.x * blockDim.x) {
      float sacc = 0.f;
      for (int l = 0; l < d.depth; ++l) sacc += p.bWo[l][d.cr_eff(l) + idx];
      p.biasS[idx] = sacc;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// conditioning: NCL fp32 (strided) <-> slab
// ------------------------------------------------------------------------------------------------
template <typename OpT>
static __global__ void __launch_bounds__(256) cond_pack_kernel(const float* __restrict__ y, long long bs, long long cs,
                                                               long long ts, int aux, int auxp, int T,
                                                               OpT* __restrict__ ycl, int is_fp16) {
  __shared__ float tile[32][33];
  int b = blockIdx.z;
  int t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int j = ty; j < 32; j += 8) {
    int c = c0 + j, t = t0 + tx;
    tile[j][tx] = (c < aux && t < T) ? y[b * bs + c * cs + t * ts] : 0.f;
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    int t = t0 + j, c = c0 + tx;
    if (t < T && c < auxp) OpTraits<OpT>::store(ycl + ((long long)b * T + t) * auxp + c, tile[tx][j], is_fp16);
  }
}

static __global__ void __launch_bounds__(256) cond_unpack_grad_kernel(const float* __restrict__ dycl, int aux, int auxp,
                                                                      int T, float* __restrict__ dy) {
  __shared__ float tile[32][33];
  int b = blockIdx.z;
  int t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int j = ty; j < 32; j += 8) {
    int t = t0 + j, c = c0 + tx;
    tile[j][tx] = (t < T && c < auxp) ? dycl[((long long)b * T + t) * auxp + c] : 0.f;
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    int c = c0 + j, t = t0 + tx;
    if (c < aux && t < T) dy[((long long)b * aux + c) * T + t] = tile[tx][j];
  }
}

// ------------------------------------------------------------------------------------------------
// tiny-K 1x1 conv from an NCL tensor to a slab:  out[row][o] = bias[o] + sum_i W[o*so + i*si] * in[b][i][t]
//   start conv   (model/waveglow.py:74,99):  in = xa (cin channels), W = start weight [Cr][cin]  (so = cin, si = 1)
//   d(end conv)  (backward of :92,105):      in = d(log_s, t) (2cin channels), W = end weight^T   (so = 1, si = Cs)
// K = 2..64 is far below a tensor-core tile, and the kernel is bound by the slab write: one thread owns
// 4 consecutive output channels of one row (16 / 8-byte stores, a warp writes contiguous rows), weights
// and the input tile sit in shared memory.  Outputs: fp32 slab and / or operand slab, optionally as a
// (hi, lo) 16-bit pair (x = hi + lo).
// ------------------------------------------------------------------------------------------------
constexpr int SMALLK_ROWS = 64;

template <typename OpT>
static __global__ void __launch_bounds__(256) smallk_to_slab_kernel(const float* __restrict__ in, long long in_bs,
                                                                    const float* __restrict__ W, int so, int si,
                                                                    const float* __restrict__ bias, int K, int C,
                                                                    int T, int blocks_per_batch, int t_off,
                                                                    int t_end, float* __restrict__ o32,
                                                                    OpT* __restrict__ ohi, OpT* __restrict__ olo,
                                                                    int is_fp16, const float* __restrict__ gscale,
                                                                    const int* __restrict__ row_len) {
  // rows [t_off, t_end) of every batch item are computed; T stays the row count of one item (strides).  row_len != nullptr:
  // rows t >= row_len[b] are written as 0 (bias included), so the slab is zero past the item's end
  extern __shared__ float sm[];
  pdl_trigger();
  pdl_wait();
  const float in_scale = gscale ? gscale[1] : 1.f;  // power-of-two gradient scale (fp16 operands), see grad_scale_kernel
  float* xs = sm;                      // [K][SMALLK_ROWS]
  float* wsm = sm + K * SMALLK_ROWS;   // [K][C]  (k-major: 4 consecutive outputs are one float4)
  const int b = blockIdx.x / blocks_per_batch;
  const int t0 = t_off + (blockIdx.x % blocks_per_batch) * SMALLK_ROWS;
  const int t_live = row_len ? row_len[b] : t_end;
  for (int idx = threadIdx.x; idx < K * SMALLK_ROWS; idx += 256) {
    int i = idx / SMALLK_ROWS, r = idx % SMALLK_ROWS;
    int t = t0 + r;
    xs[idx] = (t < t_end) ? in[b * in_bs + (long long)i * T + t] * in_scale : 0.f;
  }
  for (int idx = threadIdx.x; idx < K * C; idx += 256) {
    int i = idx / C, o = idx % C;
    wsm[idx] = W[(long long)o * so + (long long)i * si];
  }
  __syncthreads();
  if constexpr (sizeof(OpT) == 2) {
    // 16-bit slabs: 8 channels per thread, one 16-byte store per stream (a quarter warp writes one 128-byte line)
    if ((C & 7) == 0 && o32 == nullptr && ohi != nullptr) {
      const int c8 = C >> 3;
      if (K <= 8 && (256 % c8) == 0) {
        // the shapes of every shipped config (start conv: K = in_channels <= 8, d(end conv): K = 2 in_channels <= 8, 256
        // channels): a thread keeps its 8 x K weights in registers and walks the rows of its channel group
        const int o = (threadIdx.x % c8) * 8;
        float wr[8][8];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) wr[i][j] = i < K ? wsm[i * C + o + j] : 0.f;
        float bv[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) bv[j] = bias ? bias[o + j] : 0.f;
        const int rstep = 256 / c8;
        for (int r = threadIdx.x / c8; r < SMALLK_ROWS; r += rstep) {
          const int t = t0 + r;
          if (t >= t_end) break;
          float acc[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[j] = bv[j];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            if (i < K) {
              const float xv = xs[i * SMALLK_ROWS + r];
#pragma unroll
              for (int j = 0; j < 8; ++j) acc[j] = fmaf(wr[i][j], xv, acc[j]);
            }
          }
          if (t >= t_live) {
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[j] = 0.f;
          }
          const long long off = ((long long)b * T + t) * C + o;
          uint32_t h[4], l[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            h[j] = pack2(acc[2 * j], acc[2 * j + 1], is_fp16);
            float f0, f1;
            unpack2(h[j], is_fp16, f0, f1);
            l[j] = pack2(acc[2 * j] - f0, acc[2 * j + 1] - f1, is_fp16);
          }
          *reinterpret_cast<uint4*>(ohi + off) = make_uint4(h[0], h[1], h[2], h[3]);
          if (olo) *reinterpret_cast<uint4*>(olo + off) = make_uint4(l[0], l[1], l[2], l[3]);
        }
        return;
      }
      for (int idx = threadIdx.x; idx < SMALLK_ROWS * c8; idx += 256) {
        const int r = idx / c8, o = (idx % c8) * 8;
        const int t = t0 + r;
        if (t >= t_end) continue;
        float acc[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = bias ? bias[o + j] : 0.f;
        for (int i = 0; i < K; ++i) {
          const float xv = xs[i * SMALLK_ROWS + r];
          const float4 w0 = *reinterpret_cast<const float4*>(wsm + i * C + o);
          const float4 w1 = *reinterpret_cast<const float4*>(wsm + i * C + o + 4);
          acc[0] = fmaf(w0.x, xv, acc[0]); acc[1] = fmaf(w0.y, xv, acc[1]);
          acc[2] = fmaf(w0.z, xv, acc[2]); acc[3] = fmaf(w0.w, xv, acc[3]);
          acc[4] = fmaf(w1.x, xv, acc[4]); acc[5] = fmaf(w1.y, xv, acc[5]);
          acc[6] = fmaf(w1.z, xv, acc[6]); acc[7] = fmaf(w1.w, xv, acc[7]);
        }
        if (t >= t_live) {
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[j] = 0.f;
        }
        const long long off = ((long long)b * T + t) * C + o;
        uint32_t h[4], l[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          h[j] = pack2(acc[2 * j], acc[2 * j + 1], is_fp16);
          float f0, f1;
          unpack2(h[j], is_fp16, f0, f1);
          l[j] = pack2(acc[2 * j] - f0, acc[2 * j + 1] - f1, is_fp16);
        }
        *reinterpret_cast<uint4*>(ohi + off) = make_uint4(h[0], h[1], h[2], h[3]);
        if (olo) *reinterpret_cast<uint4*>(olo + off) = make_uint4(l[0], l[1], l[2], l[3]);
      }
      return;
    }
  }
  const int c4 = C >> 2;
  for (int idx = threadIdx.x; idx < SMALLK_ROWS * c4; idx += 256) {
    const int r = idx / c4, o = (idx % c4) * 4;
    const int t = t0 + r;
    if (t >= t_end) continue;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    if (bias) { acc[0] = bias[o]; acc[1] = bias[o + 1]; acc[2] = bias[o + 2]; acc[3] = bias[o + 3]; }
    for (int i = 0; i < K; ++i) {
      const float xv = xs[i * SMALLK_ROWS + r];
      const float4 w = *reinterpret_cast<const float4*>(wsm + i * C + o);
      acc[0] = fmaf(w.x, xv, acc[0]); acc[1] = fmaf(w.y, xv, acc[1]);
      acc[2] = fmaf(w.z, xv, acc[2]); acc[3] = fmaf(w.w, xv, acc[3]);
    }
    if (t >= t_live) acc[0] = acc[1] = acc[2] = acc[3] = 0.f;
    const long long off = ((long long)b * T + t) * C + o;
    if (o32) *reinterpret_cast<float4*>(o32 + off) = make_float4(acc[0], acc[1], acc[2], acc[3]);
    if constexpr (sizeof(OpT) == 4) {
      if (ohi) *reinterpret_cast<float4*>(ohi + off) = make_float4(acc[0], acc[1], acc[2], acc[3]);
    } else {
      if (ohi) {
        uint32_t h0 = pack2(acc[0], acc[1], is_fp16), h1 = pack2(acc[2], acc[3], is_fp16);
        *reinterpret_cast<uint2*>(ohi + off) = make_uint2(h0, h1);
        if (olo) {  // residual stream as hi + lo
          float f0, f1, f2, f3;
          unpack2(h0, is_fp16, f0, f1);
          unpack2(h1, is_fp16, f2, f3);
          *reinterpret_cast<uint2*>(olo + off) =
              make_uint2(pack2(acc[0] - f0, acc[1] - f1, is_fp16), pack2(acc[2] - f2, acc[3] - f3, is_fp16));
        }
      }
    }
  }
}

template <typename OpT>
static int smallk_to_slab(const float* in, long long in_bs, const float* W, int so, int si, const float* bias, int K,
                          int C, int B, int T, float* o32, OpT* ohi, OpT* olo, int is_fp16, cudaStream_t st,
                          int t_off = 0, int t_n = -1, const float* gscale = nullptr, const int* row_len = nullptr) {
  if (t_n < 0) t_n = T - t_off;
  const int bpb = ceil_div(t_n, SMALLK_ROWS);
  if (B * bpb == 0) return CMWG_OK;
  size_t smem = (size_t)K * (SMALLK_ROWS + C) * sizeof(float);
  if (smem > 48 * 1024)
    CMWG_CHECK_CUDA(cudaFuncSetAttribute(smallk_to_slab_kernel<OpT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  CMWG_CHECK_CUDA(launch_pdl(smallk_to_slab_kernel<OpT>, dim3(B * bpb), dim3(256), smem, st, in, in_bs, W, so, si, bias, K,
                             C, T, bpb, t_off, t_off + t_n, o32, ohi, olo, is_fp16, gscale, row_len));
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

// start conv backward: dx[:, :cin] += Ws^T dh0 ; block partials of dWs (and dbias)
static __global__ void __launch_bounds__(256) start_bwd_kernel(const float* __restrict__ dh0,
                                                               const uint16_t* __restrict__ dh_hi,
                                                               const uint16_t* __restrict__ dh_lo,
                                                               const float* __restrict__ x, long long x_bs,
                                                               const float* __restrict__ ws, int cin, int Cr, int T,
                                                               int blocks_per_batch, float* __restrict__ dx,
                                                               long long dx_bs, float* __restrict__ partial_w,
                                                               float* __restrict__ partial_b, int is_fp16,
                                                               const float* __restrict__ gscale) {
  extern __shared__ float sm[];
  const int LD = Cr + 1;
  const float inv_scale = gscale ? gscale[2] : 1.f;
  float* dhs = sm;                          // [32][Cr+1]
  float* xs = dhs + ROWS_PER_BLOCK * LD;    // [cin][32]
  int b = blockIdx.x / blocks_per_batch;
  int t0 = (blockIdx.x % blocks_per_batch) * ROWS_PER_BLOCK;
  for (int idx = threadIdx.x; idx < ROWS_PER_BLOCK * Cr; idx += 256) {
    int r = idx / Cr, o = idx % Cr;
    int t = t0 + r;
    float val = 0.f;
    if (t < T) {
      long long off = ((long long)b * T + t) * Cr + o;
      // tc engine: dh_0 arrives as a (hi, lo) 16-bit pair, scaled by the gradient scale
      val = dh0 ? dh0[off]
                : (op16_to_f32(dh_hi[off], is_fp16) + (dh_lo ? op16_to_f32(dh_lo[off], is_fp16) : 0.f)) * inv_scale;
    }
    dhs[r * LD + o] = val;
  }
  for (int idx = threadIdx.x; idx < cin * ROWS_PER_BLOCK; idx += 256) {
    int i = idx / ROWS_PER_BLOCK, r = idx % ROWS_PER_BLOCK;
    int t = t0 + r;
    xs[idx] = (t < T) ? x[b * x_bs + (long long)i * T + t] : 0.f;
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < cin * ROWS_PER_BLOCK; idx += 256) {
    int i = idx / ROWS_PER_BLOCK, r = idx % ROWS_PER_BLOCK;
    int t = t0 + r;
    if (t >= T) continue;
    float acc = 0.f;
    for (int o = 0; o < Cr; ++o) acc = fmaf(ws[o * cin + i], dhs[r * LD + o], acc);
    dx[b * dx_bs + (long long)i * T + t] += acc;
  }
  float* pw = partial_w + (long long)blockIdx.x * Cr * cin;
  for (int idx = threadIdx.x; idx < Cr * cin; idx += 256) {
    int o = idx / cin, i = idx % cin;
    float acc = 0.f;
    for (int r = 0; r < ROWS_PER_BLOCK; ++r) acc = fmaf(dhs[r * LD + o], xs[i * ROWS_PER_BLOCK + r], acc);
    pw[idx] = acc;
  }
  if (partial_b) {
    float* pb = partial_b + (long long)blockIdx.x * Cr;
    for (int o = threadIdx.x; o < Cr; o += 256) {
      float acc = 0.f;
      for (int r = 0; r < ROWS_PER_BLOCK; ++r) acc += dhs[r * LD + o];
      pb[o] = acc;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// 256-channel fast paths of the start / end conv backward (the shapes of every shipped config).  Both are one
// pass over a [rows][256] slab, bound by that read: a warp owns 32 consecutive rows, every lane keeps 8 channels
// (32-byte loads, a row is one fully coalesced 1 KB / 512 B request), the few "small side" values of a row (x or
// d(log_s, t): <= 8 per row) are loaded by the lane that owns the row and broadcast with shuffles, and the
// weight-gradient outer products accumulate in registers.  Warps fold into one partial per CTA in warp order and a
// CTA's row range is fixed by its index, so results are bitwise reproducible.
// ------------------------------------------------------------------------------------------------
// 8 warps x 16 rows.  (32 rows per warp left ~10 warps per SM at the LJ training shape: the per-row dependent chains -- a
// 32-byte load, CIN warp reductions -- had nothing to overlap with; measured 34 us for a 25 MB read.)
constexpr int FAST_ROWS_PER_WARP = 16;
constexpr int FAST_ROWS_PER_CTA = 8 * FAST_ROWS_PER_WARP;

__device__ __forceinline__ void load_row8(const float* __restrict__ p32, const uint16_t* __restrict__ hi,
                                          const uint16_t* __restrict__ lo, long long off, float (&v)[8],
                                          int is_fp16 = 0) {
  if (p32) {
    const float4 a = *reinterpret_cast<const float4*>(p32 + off), b = *reinterpret_cast<const float4*>(p32 + off + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  } else {
    // (hi, lo) 16-bit pair: value = hi + lo  (lo == nullptr: single-stream residual gradient, value = hi)
    const uint4 h = *reinterpret_cast<const uint4*>(hi + off);
    const uint4 l = lo ? *reinterpret_cast<const uint4*>(lo + off) : make_uint4(0u, 0u, 0u, 0u);
    const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
    if (is_fp16) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float h0, h1, l0, l1;
        unpack2(hw[j], 1, h0, h1);
        unpack2(lw[j], 1, l0, l1);
        v[2 * j] = h0 + l0;
        v[2 * j + 1] = h1 + l1;
      }
      return;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      v[2 * j] = __uint_as_float(hw[j] << 16) + __uint_as_float(lw[j] << 16);
      v[2 * j + 1] = __uint_as_float(hw[j] & 0xffff0000u) + __uint_as_float(lw[j] & 0xffff0000u);
    }
  }
}

// Sum NACC per-lane accumulators over the 8 warps of a CTA in a fixed tree order (warps 4-7 into 0-3, 2-3 into 0-1,
// 1 into 0); `buf` holds 4 * NACC * 32 floats laid out [warp][acc][lane] (conflict free).  On return warp 0 has
// stored the totals to buf[acc * 32 + lane] and the CTA is synchronised.
template <int NACC>
__device__ __forceinline__ void cta8_tree_sum(float (&acc)[NACC], float* buf) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int half = 4; half >= 1; half >>= 1) {
    if (warp >= half && warp < 2 * half) {
#pragma unroll
      for (int a = 0; a < NACC; ++a) buf[((warp - half) * NACC + a) * 32 + lane] = acc[a];
    }
    __syncthreads();
    if (warp < half) {
#pragma unroll
      for (int a = 0; a < NACC; ++a) acc[a] += buf[(warp * NACC + a) * 32 + lane];
    }
    __syncthreads();
  }
  if (warp == 0) {
#pragma unroll
    for (int a = 0; a < NACC; ++a) buf[a * 32 + lane] = acc[a];
  }
  __syncthreads();
}

// start conv backward, Cr == 256:  dx[:, i] += sum_o Ws[o][i] dh0[row][o];  partial dWs[o][i] = sum_row dh0[row][o] x[row][i]
template <int CIN>
static __global__ void __launch_bounds__(256) start_bwd256_kernel(const float* __restrict__ dh32,
                                                                  const uint16_t* __restrict__ dh_hi,
                                                                  const uint16_t* __restrict__ dh_lo,
                                                                  const float* __restrict__ x, long long x_bs,
                                                                  const float* __restrict__ ws, int TF, long long rows,
                                                                  float* __restrict__ dx, long long dx_bs,
                                                                  float* __restrict__ partial_w,
                                                                  float* __restrict__ partial_b, int is_fp16,
                                                                  const float* __restrict__ gscale) {
  __shared__ float buf[4 * (8 * CIN + 8) * 32];
  const float inv_scale = gscale ? gscale[2] : 1.f;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // acc[c * CIN + i] = dWs[lane * 8 + c][i] partial, acc[8 * CIN + c] = dbias partial
  float wreg[8][CIN], acc[8 * CIN + 8];
#pragma unroll
  for (int a = 0; a < 8 * CIN + 8; ++a) acc[a] = 0.f;
#pragma unroll
  for (int c = 0; c < 8; ++c)
#pragma unroll
    for (int i = 0; i < CIN; ++i) wreg[c][i] = ws[(lane * 8 + c) * CIN + i];
  const long long g0 = (long long)blockIdx.x * FAST_ROWS_PER_CTA + warp * FAST_ROWS_PER_WARP;
  if (g0 < rows) {
    const int nrows = (int)min((long long)FAST_ROWS_PER_WARP, rows - g0);
    const bool valid = lane < nrows;
    int b = 0, t = 0;
    if (valid) {
      b = (int)((g0 + lane) / TF);
      t = (int)((g0 + lane) - (long long)b * TF);
    }
    float xm[CIN], mine[CIN];
#pragma unroll
    for (int i = 0; i < CIN; ++i) {
      xm[i] = valid ? x[b * x_bs + (long long)i * TF + t] : 0.f;
      mine[i] = 0.f;
    }
#pragma unroll 4
    for (int r = 0; r < nrows; ++r) {
      float dh[8];
      load_row8(dh32, dh_hi, dh_lo, (g0 + r) * 256 + lane * 8, dh, is_fp16);
#pragma unroll
      for (int c = 0; c < 8; ++c) dh[c] *= inv_scale;
#pragma unroll
      for (int i = 0; i < CIN; ++i) {
        const float xv = __shfl_sync(0xffffffffu, xm[i], r);
        float p = 0.f;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          acc[c * CIN + i] = fmaf(dh[c], xv, acc[c * CIN + i]);
          p = fmaf(wreg[c][i], dh[c], p);
        }
        p = warp_sum(p);
        if (lane == r) mine[i] = p;
      }
#pragma unroll
      for (int c = 0; c < 8; ++c) acc[8 * CIN + c] += dh[c];
    }
    if (valid) {
#pragma unroll
      for (int i = 0; i < CIN; ++i) dx[b * dx_bs + (long long)i * TF + t] += mine[i];
    }
  }
  cta8_tree_sum<8 * CIN + 8>(acc, buf);
  float* pw = partial_w + (long long)blockIdx.x * 256 * CIN;
  for (int idx = threadIdx.x; idx < 256 * CIN; idx += 256) {
    const int o = idx / CIN, i = idx - o * CIN;
    pw[idx] = buf[((o & 7) * CIN + i) * 32 + (o >> 3)];
  }
  if (partial_b)
    partial_b[(long long)blockIdx.x * 256 + threadIdx.x] = buf[(8 * CIN + (threadIdx.x & 7)) * 32 + (threadIdx.x >> 3)];
}

// end conv weight gradient, Cs == 256:  partial dWe[oc][k] = sum_row dlst[b][oc][t] skip[row][k];  dbias[oc] = sum dlst
template <int COUT>
static __global__ void __launch_bounds__(256) end_bwd_dw256_kernel(const float* __restrict__ dlst,
                                                                   const float* __restrict__ skip, int TF,
                                                                   long long rows, float* __restrict__ partial_w,
                                                                   float* __restrict__ partial_b) {
  __shared__ float buf[4 * (8 * COUT + COUT) * 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // acc[oc * 8 + c] = dWe[oc][lane * 8 + c] partial, acc[8 * COUT + oc] = this lane's share of dbias[oc]
  float acc[8 * COUT + COUT];
#pragma unroll
  for (int a = 0; a < 8 * COUT + COUT; ++a) acc[a] = 0.f;
  const long long g0 = (long long)blockIdx.x * FAST_ROWS_PER_CTA + warp * FAST_ROWS_PER_WARP;
  if (g0 < rows) {
    const int nrows = (int)min((long long)FAST_ROWS_PER_WARP, rows - g0);
    float dl[COUT];
    if (lane < nrows) {
      const int b = (int)((g0 + lane) / TF);
      const int t = (int)((g0 + lane) - (long long)b * TF);
#pragma unroll
      for (int oc = 0; oc < COUT; ++oc) dl[oc] = dlst[((long long)b * COUT + oc) * TF + t];
    } else {
#pragma unroll
      for (int oc = 0; oc < COUT; ++oc) dl[oc] = 0.f;
    }
#pragma unroll
    for (int oc = 0; oc < COUT; ++oc) acc[8 * COUT + oc] = dl[oc];
#pragma unroll 4
    for (int r = 0; r < nrows; ++r) {
      float sk[8];
      load_row8(skip, nullptr, nullptr, (g0 + r) * 256 + lane * 8, sk);
#pragma unroll
      for (int oc = 0; oc < COUT; ++oc) {
        const float v = __shfl_sync(0xffffffffu, dl[oc], r);
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[oc * 8 + c] = fmaf(v, sk[c], acc[oc * 8 + c]);
      }
    }
  }
  cta8_tree_sum<8 * COUT + COUT>(acc, buf);
  float* pw = partial_w + (long long)blockIdx.x * COUT * 256;
  for (int idx = threadIdx.x; idx < COUT * 256; idx += 256) {
    const int oc = idx >> 8, k = idx & 255;
    pw[idx] = buf[(oc * 8 + (k & 7)) * 32 + (k >> 3)];
  }
  if (partial_b && threadIdx.x < COUT * 32) {
    // one warp per output channel folds the 32 lane shares in shuffle order
    const float sb = warp_sum(buf[(8 * COUT + warp) * 32 + lane]);
    if (lane == 0) partial_b[(long long)blockIdx.x * COUT + warp] = sb;
  }
}

// ------------------------------------------------------------------------------------------------
// end conv (Cs -> 2cin, kernel 1): slab fp32 input, NCL output          model/waveglow.py:92,105
// Bound by the read of the fp32 skip slab.  One warp owns 32 consecutive time steps: per row every lane
// loads KV float4 (a fully coalesced row), multiplies with its register-resident weight slice for up
// to 8 output channels, the partials are summed with xor-shuffles (fixed order: deterministic), and lane
// r keeps row r's results so that the final NCL stores are 128-byte coalesced.
// ------------------------------------------------------------------------------------------------
template <int KV>
static __global__ void __launch_bounds__(128) end_fwd_kernel(const float* __restrict__ skip,
                                                             const float* __restrict__ we,
                                                             const float* __restrict__ bias, int cout, int Cs, int T,
                                                             int B, int t_off, int t_n, float* __restrict__ lst) {
  // rows [t_off, t_off + t_n) of every batch item; T is the row count of one item (strides)
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int wpb = (t_n + 31) >> 5;
  const int gw = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (gw >= B * wpb) return;
  const int b = gw / wpb, t0 = t_off + (gw % wpb) * 32;
  const int nrows = min(32, t_off + t_n - t0);
  const float* base = skip + ((long long)b * T + t0) * Cs;
  for (int oc0 = 0; oc0 < cout; oc0 += 8) {
    float4 w[8][KV];
#pragma unroll
    for (int c = 0; c < 8; ++c)
#pragma unroll
      for (int j = 0; j < KV; ++j) {
        int k = 4 * lane + 128 * j;
        w[c][j] = (oc0 + c < cout && k < Cs) ? *reinterpret_cast<const float4*>(we + (long long)(oc0 + c) * Cs + k)
                                             : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    float mine[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) mine[c] = (bias && oc0 + c < cout) ? bias[oc0 + c] : 0.f;
#pragma unroll 4
    for (int r = 0; r < nrows; ++r) {
      float4 sv[KV];
#pragma unroll
      for (int j = 0; j < KV; ++j) {
        int k = 4 * lane + 128 * j;
        sv[j] = (k < Cs) ? *reinterpret_cast<const float4*>(base + (long long)r * Cs + k) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        float p = 0.f;
#pragma unroll
        for (int j = 0; j < KV; ++j) {
          p = fmaf(w[c][j].x, sv[j].x, p); p = fmaf(w[c][j].y, sv[j].y, p);
          p = fmaf(w[c][j].z, sv[j].z, p); p = fmaf(w[c][j].w, sv[j].w, p);
        }
        p = warp_sum(p);
        if (lane == r) mine[c] += p;
      }
    }
    if (lane < nrows) {
#pragma unroll
      for (int c = 0; c < 8; ++c)
        if (oc0 + c < cout) lst[((long long)b * cout + oc0 + c) * T + t0 + lane] = mine[c];
    }
  }
}

static int end_fwd_launch(const float* skip, const float* we, const float* bias, int cout, int Cs, int B, int T,
                          float* lst, cudaStream_t st, int t_off = 0, int t_n = -1) {
  if (t_n < 0) t_n = T - t_off;
  const int warps = B * ceil_div(t_n, 32);
  const int grid = ceil_div(warps, 4);
  if (grid == 0) return CMWG_OK;
  const int kv = ceil_div(Cs, 128);
  CMWG_REQUIRE(kv <= 4, "end conv: skip_channels %d > 512 not supported", Cs);
  if (kv == 1)
    CMWG_CHECK_CUDA(launch_pdl(end_fwd_kernel<1>, dim3(grid), dim3(128), 0, st, skip, we, bias, cout, Cs, T, B, t_off, t_n, lst));
  else if (kv == 2)
    CMWG_CHECK_CUDA(launch_pdl(end_fwd_kernel<2>, dim3(grid), dim3(128), 0, st, skip, we, bias, cout, Cs, T, B, t_off, t_n, lst));
  else
    CMWG_CHECK_CUDA(launch_pdl(end_fwd_kernel<4>, dim3(grid), dim3(128), 0, st, skip, we, bias, cout, Cs, T, B, t_off, t_n, lst));
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

static __global__ void __launch_bounds__(256) end_bwd_dw_kernel(const float* __restrict__ dlst,
                                                                const float* __restrict__ skip, int cout, int Cs,
                                                                int T, int blocks_per_batch,
                                                                float* __restrict__ partial_w,
                                                                float* __restrict__ partial_b) {
  extern __shared__ float sm[];
  float* dl = sm;                           // [cout][32]
  float* sk = sm + cout * ROWS_PER_BLOCK;   // [32][Cs]
  int b = blockIdx.x / blocks_per_batch;
  int t0 = (blockIdx.x % blocks_per_batch) * ROWS_PER_BLOCK;
  for (int idx = threadIdx.x; idx < cout * ROWS_PER_BLOCK; idx += 256) {
    int oc = idx / ROWS_PER_BLOCK, r = idx % ROWS_PER_BLOCK;
    int t = t0 + r;
    dl[idx] = (t < T) ? dlst[((long long)b * cout + oc) * T + t] : 0.f;
  }
  for (int idx = threadIdx.x; idx < ROWS_PER_BLOCK * Cs; idx += 256) {
    int r = idx / Cs, k = idx % Cs;
    int t = t0 + r;
    sk[idx] = (t < T) ? skip[((long long)b * T + t) * Cs + k] : 0.f;
  }
  __syncthreads();
  float* pw = partial_w + (long long)blockIdx.x * cout * Cs;
  for (int idx = threadIdx.x; idx < cout * Cs; idx += 256) {
    int oc = idx / Cs, k = idx % Cs;
    float acc = 0.f;
    for (int r = 0; r < ROWS_PER_BLOCK; ++r) acc = fmaf(dl[oc * ROWS_PER_BLOCK + r], sk[r * Cs + k], acc);
    pw[idx] = acc;
  }
  if (partial_b) {
    float* pb = partial_b + (long long)blockIdx.x * cout;
    for (int oc = threadIdx.x; oc < cout; oc += 256) {
      float acc = 0.f;
      for (int r = 0; r < ROWS_PER_BLOCK; ++r) acc += dl[oc * ROWS_PER_BLOCK + r];
      pb[oc] = acc;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Gradient scaling for fp16 operands.  fp16 carries the same 10 mantissa bits as TF32 (bf16: 7) at bf16's tensor-core rate,
// but only 5 exponent bits; the backward GEMM chain is LINEAR in the incoming cotangent, so it runs on S * cotangent with S a
// power of two chosen per call on the device (no host round trip), and every result is multiplied by 1 / S where it leaves
// the 16-bit slabs (exact: powers of two).  gscale = {max |dlst| (bit pattern), S, 1 / S, arrival counter}.
//   S = 2^(8 - ceil(log2(max|dlst| * max_k sum_o |W_end[o][k]|)))  =>  |S * dskip| <= 256:
// 2^8 of headroom below fp16's largest value for the growth of the residual gradient through the layers, and 2^22 of normal
// range below the largest entry (smaller entries lose precision gradually as fp16 subnormals; they do not matter to any norm).
// ------------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(256) grad_scale_kernel(float* __restrict__ gscale, const float* __restrict__ dlst,
                                                                long long n, const float* __restrict__ w_end, int cout,
                                                                int Cs) {
  // gscale[0] (bit pattern of the running max) and gscale[3] (arrival counter) are zeroed by the caller.  Every CTA folds its
  // slice of dlst into the max (order independent: deterministic); the last CTA to arrive forms the bound and the scale.
  __shared__ float red[8];
  __shared__ bool last;
  float m = 0.f;
  const long long n4 = n >> 2;
  const float4* a4 = reinterpret_cast<const float4*>(dlst);
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < n4; i += (long long)gridDim.x * 256) {
    const float4 v = a4[i];
    m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
  }
  if (blockIdx.x == 0)
    for (long long i = (n4 << 2) + threadIdx.x; i < n; i += 256) m = fmaxf(m, fabsf(dlst[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < 8; ++i) m = fmaxf(m, red[i]);
    if (m > 0.f) atomicMax(reinterpret_cast<unsigned int*>(gscale), __float_as_uint(m));  // non-negative floats order like their bits
    __threadfence();
    last = atomicAdd(reinterpret_cast<unsigned int*>(gscale) + 3, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  float colmax = 0.f;
  for (int k = threadIdx.x; k < Cs; k += 256) {
    float s = 0.f;
    for (int o = 0; o < cout; ++o) s += fabsf(w_end[(long long)o * Cs + k]);
    colmax = fmaxf(colmax, s);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) colmax = fmaxf(colmax, __shfl_xor_sync(0xffffffffu, colmax, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = colmax;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < 8; ++i) colmax = fmaxf(colmax, red[i]);
    const float amax = __uint_as_float(*reinterpret_cast<volatile unsigned int*>(gscale));
    const float bound = colmax * amax;
    float S = 1.f;
    if (bound > 0.f && bound < 3.0e38f) {
      int e = 8 - (int)ceilf(log2f(bound));
      // S * dlst itself is an fp16 operand when the `end` conv is folded into the dgate GEMM (dl_slab_kernel): keep it
      // below 2^14 (only a nearly-zero `end` weight makes this the binding bound)
      e = min(e, 14 - (int)ceilf(log2f(amax)));
      e = max(-60, min(60, e));
      S = exp2f((float)e);
    }
    gscale[1] = S;
    gscale[2] = 1.f / S;
  }
}

// in-place multiply by gscale[idx] (fp32 buffers that leave the scaled domain without passing another kernel)
static __global__ void __launch_bounds__(256) scale_by_kernel(float* __restrict__ a, long long n4,
                                                              const float* __restrict__ gscale, int idx) {
  const float sc = gscale[idx];
  float4* p = reinterpret_cast<float4*>(a);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 v = p[i];
    v.x *= sc; v.y *= sc; v.z *= sc; v.w *= sc;
    p[i] = v;
  }
}

// ------------------------------------------------------------------------------------------------
// reductions
// ------------------------------------------------------------------------------------------------
// out[p] = sum_j partial[j][p] in a fixed order: a CTA owns 32 outputs, its 8 warps take the partials j = y, y + 8, ... (fp64),
// and the eight sub-sums are folded in warp order.  Reads are 128-byte rows of 32 consecutive outputs.
static __global__ void __launch_bounds__(256) reduce_blocks_kernel(const float* __restrict__ partial, int nblocks,
                                                                   int P, float* __restrict__ out,
                                                                   const float* __restrict__ gscale) {
  __shared__ double part[8][32];
  const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
  const int p = blockIdx.x * 32 + x;
  double s = 0.0;
  if (p < P)
    for (int j = y; j < nblocks; j += 8) s += (double)partial[(long long)j * P + p];
  part[y][x] = s;
  __syncthreads();
  if (y == 0 && p < P) {
    double t = part[0][x];
#pragma unroll
    for (int k = 1; k < 8; ++k) t += part[k][x];
    out[p] = (float)t * (gscale ? gscale[2] : 1.f);
  }
}

// split-K partials [splits][M][N] of several weight-gradient problems -> strided destinations
struct WgReduceEntry {
  const float* partial;
  int splits;            // partial tiles to sum
  int M, N, n_valid;     // stored dims, valid columns
  float* out;
  long long sm, sn, off; // out[off + m*sm + n*sn]
};
struct WgReduceTable {
  WgReduceEntry e[TC_MAX_WG_REDUCE];
  int n;
  const float* gscale;   // nullptr, or the gradient-scale triple: results are multiplied by gscale[2] = 1 / S
};

static __global__ void __launch_bounds__(256) wgrad_reduce_kernel(const WgReduceTable tb) {
  const WgReduceEntry& e = tb.e[blockIdx.y];
  const float inv_scale = tb.gscale ? tb.gscale[2] : 1.f;
  const int nv4 = (e.n_valid + 3) >> 2;  // stored N is a multiple of 4, so the float4 loads stay in bounds
  long long total = (long long)e.M * nv4;
  const long long stride = (long long)e.M * e.N;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    int m = (int)(idx / nv4), n = (int)(idx % nv4) * 4;
    const float* p = e.partial + (long long)m * e.N + n;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    int j = 0;
    for (; j + 4 <= e.splits; j += 4) {  // four loads in flight, summed in split order: deterministic
      const float4 v0 = *reinterpret_cast<const float4*>(p + j * stride);
      const float4 v1 = *reinterpret_cast<const float4*>(p + (j + 1) * stride);
      const float4 v2 = *reinterpret_cast<const float4*>(p + (j + 2) * stride);
      const float4 v3 = *reinterpret_cast<const float4*>(p + (j + 3) * stride);
      s.x += v0.x; s.y += v0.y; s.z += v0.z; s.w += v0.w;
      s.x += v1.x; s.y += v1.y; s.z += v1.z; s.w += v1.w;
      s.x += v2.x; s.y += v2.y; s.z += v2.z; s.w += v2.w;
      s.x += v3.x; s.y += v3.y; s.z += v3.z; s.w += v3.w;
    }
    if (j + 2 <= e.splits) {
      const float4 v0 = *reinterpret_cast<const float4*>(p + j * stride);
      const float4 v1 = *reinterpret_cast<const float4*>(p + (j + 1) * stride);
      s.x += v0.x; s.y += v0.y; s.z += v0.z; s.w += v0.w;
      s.x += v1.x; s.y += v1.y; s.z += v1.z; s.w += v1.w;
      j += 2;
    }
    if (j < e.splits) {
      const float4 v = *reinterpret_cast<const float4*>(p + j * stride);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    float* o = e.out + e.off + m * e.sm + n * e.sn;
    o[0] = s.x * inv_scale;
    if (n + 1 < e.n_valid) o[e.sn] = s.y * inv_scale;
    if (n + 2 < e.n_valid) o[2 * e.sn] = s.z * inv_scale;
    if (n + 3 < e.n_valid) o[3 * e.sn] = s.w * inv_scale;
  }
}

// two-level fixed-order reduction of block partials: [nblocks][P] -> [ceil(nblocks/64)][P]
static __global__ void __launch_bounds__(128) reduce_blocks_stage_kernel(const float* __restrict__ partial, int nblocks,
                                                                         int P, float* __restrict__ out) {
  int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  int j0 = blockIdx.y * 64, j1 = min(j0 + 64, nblocks);
  float s = 0.f;
  for (int j = j0; j < j1; ++j) s += partial[(long long)j * P + p];
  out[(long long)blockIdx.y * P + p] = s;
}

// out[b][j] = sum_h in[b][h][j] (fixed order), j in float4 units: per-line conditioning gradient -> (B, T, auxp)
static __global__ void __launch_bounds__(256) sum_lines_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                               int H, long long n4) {
  const int b = blockIdx.y;
  const float4* src = reinterpret_cast<const float4*>(in) + (long long)b * H * n4;
  float4* dst = reinterpret_cast<float4*>(out) + (long long)b * n4;
  for (long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x; j < n4; j += (long long)gridDim.x * blockDim.x) {
    float4 s = src[j];
    for (int h = 1; h < H; ++h) {
      float4 v = src[(long long)h * n4 + j];
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    dst[j] = s;
  }
}

// column sums of a slab (bias gradients): block partials over 32 rows
template <typename OpT>
static __global__ void __launch_bounds__(256) colsum_partial_kernel(const OpT* __restrict__ a, int ld, int C,
                                                                    long long rows, float* __restrict__ partial,
                                                                    int is_fp16) {
  long long r0 = (long long)blockIdx.x * ROWS_PER_BLOCK;
  for (int c = threadIdx.x; c < C; c += 256) {
    float acc = 0.f;
    for (int r = 0; r < ROWS_PER_BLOCK; ++r) {
      long long row = r0 + r;
      if (row < rows) acc += OpTraits<OpT>::load(a + row * ld + c, is_fp16);
    }
    partial[(long long)blockIdx.x * C + c] = acc;
  }
}

}  // namespace cmwg
