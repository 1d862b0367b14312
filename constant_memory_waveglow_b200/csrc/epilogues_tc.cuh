// Epilogue functors of the tcgen05 engine.  One call covers ONE accumulator row (= one (batch, time)
// column of the reference's NCL tensors) and 16 consecutive epilogue columns; inputs and outputs are
// register fragments that the engine moves through swizzled shared-memory staging and TMA.
//
//   kPaired    the tile's columns [0, BN/2) and [BN/2, BN) are partner pre-activations (tanh / sigmoid)
//   kOut       output streams (each a slab the engine TMA-stores 32 rows x 32 columns at a time)
//   kOutF32    outputs are fp32 (else 16-bit operands, two per register)
//   kOutBufs   staging buffers per output stream (2 = the store of chunk i overlaps chunk i+1)
//   kIn        16-bit input streams, TMA-loaded one chunk ahead
//   kColGroups epilogue warps per TMEM lane quadrant (4: shortest epilogue; 2: half the staging, more
//              operand stages -- for GEMMs whose K loop is long enough to hide a longer epilogue)
//   out_col(i, c0) / in_col(i, c0)   channel coordinate of stream i for epilogue column c0
// Precision / bias switches are warp-uniform branches AROUND the unrolled loops (never per element),
// so only one variant's instructions are issued.
#pragma once
#include "epilogues.cuh"

namespace cmwg {

// ---- gate: g = tanh(pre_t) * sigmoid(pre_s)  (model/waveglow.py:13-15,42-44) ---------------------
// SAVE additionally stores sigmoid(pre_s) for the backward pass.  tanh(pre_t) is NOT stored: the backward recovers it as
// g / sigmoid (GateBwdTcEpi), so a saving gate tile writes two 16-bit streams instead of three -- both fit the two staging
// buffers of an epilogue warp at once (no wait for the first stores before the third stream can be staged) and a WN
// forward with saves writes 25 % fewer bytes.
template <bool SAVE>
struct GateTcEpi {
  static constexpr bool kPaired = true, kOutF32 = false;
  static constexpr int kOut = SAVE ? 2 : 1, kIn = 0, kOutBufs = 1, kColGroups = 4;
  const float* bias;  // nullptr or [2][Cd]
  int Cd, f16;
  __device__ __forceinline__ int out_col(int, int c0) const { return c0; }
  __device__ __forceinline__ int in_col(int, int c0) const { return c0; }
  __device__ __forceinline__ void compute(int ch0, float (&lo)[16], float (&hi)[16], uint32_t (&o)[kOut][8]) const {
    if (bias) {
#pragma unroll
      for (int j = 0; j < 16; ++j) { lo[j] += __ldg(bias + ch0 + j); hi[j] += __ldg(bias + Cd + ch0 + j); }
    }
    if (f16) {
      // fp16's 11-bit mantissa deserves better than tanh.approx (2^-11 relative error): exact-to-1e-7 forms on
      // MUFU.EX2 / MUFU.RCP, three MUFU operations per gate value (the MUFU pipe runs 16 lanes per clock per SM, a
      // quarter of an epilogue's budget at four) -- see gate_ex2()
#pragma unroll
      for (int j = 0; j < 16; j += 2) {
        float a0, b0, g0, a1, b1, g1;
        gate_ex2<SAVE>(lo[j], hi[j], a0, b0, g0);
        gate_ex2<SAVE>(lo[j + 1], hi[j + 1], a1, b1, g1);
        o[0][j >> 1] = pack2(g0, g1, 1);
        if constexpr (SAVE) o[1][j >> 1] = pack2(b0, b1, 1);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 16; j += 2) {
        float a0 = tanh_f<true>(lo[j]), a1 = tanh_f<true>(lo[j + 1]);
        float b0 = sigmoid_f<true>(hi[j]), b1 = sigmoid_f<true>(hi[j + 1]);
        o[0][j >> 1] = pack2(a0 * b0, a1 * b1, 0);
        if constexpr (SAVE) o[1][j >> 1] = pack2(b0, b1, 0);
      }
    }
  }
};

// ---- (hi, lo) split store with optional (hi, lo) addend ------------------------------------------
// The tcgen05 pipeline keeps the residual stream (and its gradient) as a PAIR of 16-bit slabs,
// x = hi + lo with hi = rn16(x), lo = rn16(x - hi) (precision of the pair: 2^-17 relative); hi doubles
// as the GEMM operand of the next dilated conv.  ADD: out = acc + in_hi + in_lo, the residual add of
// model/waveglow.py:46 (forward) or the upstream residual gradient (backward), summed in fp32.
template <bool ADD, int CG = 4>
struct SplitTcEpi {
  static constexpr bool kPaired = false, kOutF32 = false;
  static constexpr int kOut = 2, kIn = ADD ? 2 : 0, kOutBufs = 1, kColGroups = CG;
  const float* bias;
  int f16;
  __device__ __forceinline__ int out_col(int, int c0) const { return c0; }
  __device__ __forceinline__ int in_col(int, int c0) const { return c0; }
  template <int F16>
  __device__ __forceinline__ void split(const float (&x)[16], uint32_t (&o)[2][8]) const {
#pragma unroll
    for (int j = 0; j < 16; j += 2) {
      uint32_t h = pack2(x[j], x[j + 1], F16);
      float h0, h1;
      unpack2(h, F16, h0, h1);
      o[0][j >> 1] = h;
      o[1][j >> 1] = pack2(x[j] - h0, x[j + 1] - h1, F16);
    }
  }
  __device__ __forceinline__ void add_bias(int col0, float (&x)[16]) const {
    if (bias) {
#pragma unroll
      for (int j = 0; j < 16; ++j) x[j] += __ldg(bias + col0 + j);
    }
  }
  __device__ __forceinline__ void compute(int col0, float (&v)[16], uint32_t (&o)[2][8]) const {
    add_bias(col0, v);
    if (f16) split<1>(v, o);
    else split<0>(v, o);
  }
  __device__ __forceinline__ void compute(int col0, float (&v)[16], const uint32_t (&in)[2][8],
                                          uint32_t (&o)[2][8]) const {
    add_bias(col0, v);
    if (f16) {
#pragma unroll
      for (int j = 0; j < 16; j += 2) {
        float h0, h1, l0, l1;
        unpack2(in[0][j >> 1], 1, h0, h1);
        unpack2(in[1][j >> 1], 1, l0, l1);
        v[j] += h0 + l0;
        v[j + 1] += h1 + l1;
      }
      split<1>(v, o);
    } else {
#pragma unroll
      for (int j = 0; j < 16; j += 2) {
        float h0, h1, l0, l1;
        unpack2(in[0][j >> 1], 0, h0, h1);
        unpack2(in[1][j >> 1], 0, l0, l1);
        v[j] += h0 + l0;
        v[j + 1] += h1 + l1;
      }
      split<0>(v, o);
    }
  }
};

// ---- residual add on ONE 16-bit stream: out = rn16(acc + in) ---------------------------------------
// fp16 operands: the residual stream (forward) and its gradient (backward) are carried as the operand slab alone.  The extra rounding per layer
// (2^-12 relative, on a stream every dilated conv re-reads rounded to fp16 anyway) measures as +20 % on the error of the WN
// output (profiles/r02_precision.json), and a residual tile moves half the bytes: its whole input fits the warp's two staging
// buffers, so nothing is loaded while the accumulator waits.  bf16 operands (8 mantissa bits) keep the (hi, lo) pair.
template <int CG = 4>
struct AddTcEpiT {
  static constexpr bool kPaired = false, kOutF32 = false;
  static constexpr int kOut = 1, kIn = 1, kOutBufs = 1, kColGroups = CG;
  const float* bias;
  int f16;
  __device__ __forceinline__ int out_col(int, int c0) const { return c0; }
  __device__ __forceinline__ int in_col(int, int c0) const { return c0; }
  __device__ __forceinline__ void compute(int col0, float (&v)[16], const uint32_t (&in)[1][8], uint32_t (&o)[1][8]) const {
    if (bias) {
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] += __ldg(bias + col0 + j);
    }
    if (f16) {
#pragma unroll
      for (int j = 0; j < 16; j += 2) {
        float h0, h1;
        unpack2(in[0][j >> 1], 1, h0, h1);
        o[0][j >> 1] = pack2(v[j] + h0, v[j + 1] + h1, 1);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 16; j += 2) {
        float h0, h1;
        unpack2(in[0][j >> 1], 0, h0, h1);
        o[0][j >> 1] = pack2(v[j] + h0, v[j + 1] + h1, 0);
      }
    }
  }
};

using AddTcEpi = AddTcEpiT<4>;

// ---- plain 16-bit store: out = rn16(acc)  (first tile of a single-stream chain: nothing to add) ----
struct RoundTcEpi {
  static constexpr bool kPaired = false, kOutF32 = false;
  static constexpr int kOut = 1, kIn = 0, kOutBufs = 1, kColGroups = 4;
  int f16;
  __device__ __forceinline__ int out_col(int, int c0) const { return c0; }
  __device__ __forceinline__ int in_col(int, int c0) const { return c0; }
  __device__ __forceinline__ void compute(int, float (&v)[16], uint32_t (&o)[1][8]) const {
    if (f16) {
#pragma unroll
      for (int j = 0; j < 16; j += 2) o[0][j >> 1] = pack2(v[j], v[j + 1], 1);
    } else {
#pragma unroll
      for (int j = 0; j < 16; j += 2) o[0][j >> 1] = pack2(v[j], v[j + 1], 0);
    }
  }
};

// ---- gate backward: dpre = dg * d(tanh * sigmoid) ------------------------------------------------
// inputs: the gate output g = tanh * sigmoid and the saved sigmoid (both 16-bit slabs of the recompute); tanh = g / sigmoid
// (one MUFU.RCP; where the sigmoid has underflowed to 0 so has g, and both gradient halves carry a factor sigmoid = 0);
// outputs: the tanh-half and sigmoid-half gradients, columns [0, Cd) and [Cd, 2Cd) of the dpre slab (two tensor maps, one
// per column window).  With fp16 operands the accumulator holds S * dg (gradient scale, wn_kernels.cuh); the functor is
// linear in it.
__device__ __forceinline__ float tanh_from_gate(float g, float s) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(fmaxf(s, 5.9604645e-8f)));   // smallest fp16 subnormal: s = 0 -> g = 0 -> 0
  return fminf(fmaxf(g * r, -1.f), 1.f);
}
struct GateBwdTcEpi {
  static constexpr bool kPaired = false, kOutF32 = false;
  static constexpr int kOut = 2, kIn = 2, kOutBufs = 1, kColGroups = 4;
  int f16;
  __device__ __forceinline__ int out_col(int, int c0) const { return c0; }
  __device__ __forceinline__ int in_col(int, int c0) const { return c0; }
  template <int F16>
  __device__ __forceinline__ void run(float (&v)[16], const uint32_t (&in)[2][8], uint32_t (&o)[2][8]) const {
#pragma unroll
    for (int j = 0; j < 16; j += 2) {
      float g0, g1, b0, b1;
      unpack2(in[0][j >> 1], F16, g0, g1);
      unpack2(in[1][j >> 1], F16, b0, b1);
      const float a0 = tanh_from_gate(g0, b0), a1 = tanh_from_gate(g1, b1);
      float t0 = v[j] * b0, t1 = v[j + 1] * b1;  // dg * sigmoid
      o[0][j >> 1] = pack2(t0 * (1.f - a0 * a0), t1 * (1.f - a1 * a1), F16);
      o[1][j >> 1] = pack2(t0 * a0 * (1.f - b0), t1 * a1 * (1.f - b1), F16);
    }
  }
  __device__ __forceinline__ void compute(int, float (&v)[16], const uint32_t (&in)[2][8], uint32_t (&o)[2][8]) const {
    if (f16) run<1>(v, in, o);
    else run<0>(v, in, o);
  }
};

// ---- plain fp32 store (skip sum, conditioning gradient, self tests) -------------------------------
struct StoreTcEpi {
  static constexpr bool kPaired = false, kOutF32 = true;
  static constexpr int kOut = 1, kIn = 0, kOutBufs = 1, kColGroups = 4;
  const float* bias;    // nullptr or [N]
  const float* gscale;  // nullptr, or the gradient-scale triple: the accumulator is multiplied by gscale[2] = 1 / S
  __device__ __forceinline__ int out_col(int, int c0) const { return c0; }
  __device__ __forceinline__ int in_col(int, int c0) const { return c0; }
  __device__ __forceinline__ void compute(int col0, float (&v)[16], uint32_t (&o)[1][16]) const {
    if (gscale) {
      const float sc = __ldg(gscale + 2);
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] *= sc;
    }
    if (bias) {
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] += __ldg(bias + col0 + j);
    }
#pragma unroll
    for (int j = 0; j < 16; ++j) o[0][j] = __float_as_uint(v[j]);
  }
};

}  // namespace cmwg
