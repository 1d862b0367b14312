// Epilogue functors shared by the FFMA engine and the tcgen05 engine.  Each call covers one output
// ROW (= one (batch, time) column of the reference's NCL tensors) and NC consecutive channels, so
// every global access is NC*sizeof contiguous.
//
// Two-phase interface (the tcgen05 engine keeps 8 fragments in flight per lane):
//   load<NC>(row, col0, aux)            global reads the epilogue needs (residual, skip, saved gate values)
//   apply<NC>(row, col0, acc, aux)      arithmetic + global writes
// op<NC>(row, col0, acc) = load + apply (used by the FFMA engine).  kAux = floats of `aux` per column.
#pragma once
#include "common.cuh"

namespace cmwg {

// two floats -> one packed 16-bit pair with a single cvt.rn.{bf16x2,f16x2}.f32
__device__ __forceinline__ uint32_t pack2(float lo, float hi, int f16) {
  if (f16) {
    // one F2FP.SATFINITE.F16.F32.PACK_AB: round to nearest even, +-65504 instead of inf beyond fp16's range
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
  }
  __nv_bfloat162 b = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&b);
}
__device__ __forceinline__ void unpack2(uint32_t u, int f16, float& lo, float& hi) {
  if (f16) {
    float2 f = __half22float2(*reinterpret_cast<__half2*>(&u));
    lo = f.x; hi = f.y;
  } else {
    lo = __uint_as_float(u << 16);
    hi = __uint_as_float(u & 0xffff0000u);
  }
}

template <typename OpT, int NC>
__device__ __forceinline__ void store_ops(OpT* dst, const float* v, int f16) {
  if constexpr (sizeof(OpT) == 4) {
#pragma unroll
    for (int j = 0; j < NC; j += 4)
      *reinterpret_cast<float4*>(dst + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
  } else {
    if constexpr (NC % 8 == 0) {
#pragma unroll
      for (int j = 0; j < NC; j += 8) {
        uint4 u;
        u.x = pack2(v[j + 0], v[j + 1], f16);
        u.y = pack2(v[j + 2], v[j + 3], f16);
        u.z = pack2(v[j + 4], v[j + 5], f16);
        u.w = pack2(v[j + 6], v[j + 7], f16);
        *reinterpret_cast<uint4*>(dst + j) = u;
      }
    } else {
#pragma unroll
      for (int j = 0; j < NC; j += 4) {
        uint2 u;
        u.x = pack2(v[j + 0], v[j + 1], f16);
        u.y = pack2(v[j + 2], v[j + 3], f16);
        *reinterpret_cast<uint2*>(dst + j) = u;
      }
    }
  }
}

template <typename OpT, int NC>
__device__ __forceinline__ void load_ops(const OpT* src, float* v, int f16) {
  if constexpr (sizeof(OpT) == 4) {
#pragma unroll
    for (int j = 0; j < NC; j += 4) {
      float4 q = *reinterpret_cast<const float4*>(src + j);
      v[j] = q.x; v[j + 1] = q.y; v[j + 2] = q.z; v[j + 3] = q.w;
    }
  } else {
#pragma unroll
    for (int j = 0; j < NC; j += 4) {
      uint2 u = *reinterpret_cast<const uint2*>(src + j);
      unpack2(u.x, f16, v[j + 0], v[j + 1]);
      unpack2(u.y, f16, v[j + 2], v[j + 3]);
    }
  }
}

template <int NC>
__device__ __forceinline__ void load_f32(const float* src, float* v) {
#pragma unroll
  for (int j = 0; j < NC; j += 4) {
    float4 q = *reinterpret_cast<const float4*>(src + j);
    v[j] = q.x; v[j + 1] = q.y; v[j + 2] = q.z; v[j + 3] = q.w;
  }
}
template <int NC>
__device__ __forceinline__ void store_f32(float* dst, const float* v) {
#pragma unroll
  for (int j = 0; j < NC; j += 4) *reinterpret_cast<float4*>(dst + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
}

// ---- 1. gate: g = tanh(pre_t) * sigmoid(pre_s)  (model/waveglow.py:13-15,42-44) -----------------
// The gate GEMM's weight rows are permuted so that the partner pre-activations of gate channel ch
// sit G columns apart inside one N tile; the engine hands both halves to pair().
template <typename OpT, bool FAST>
struct GateEpi {
  OpT* g;          // [rows][Cd]
  OpT* a_save;     // [rows][Cd] or nullptr: tanh(pre_t)   (kept for the backward)
  OpT* b_save;     // [rows][Cd] or nullptr: sigmoid(pre_s)
  const float* bias;  // nullptr or [2][Cd]
  int Cd;
  int f16;
  template <int NC>
  __device__ __forceinline__ void pair(long long row, int ch0, const float (&lo)[NC], const float (&hi)[NC]) const {
    if (ch0 >= Cd) return;  // Cd % 4 == 0 and NC | (Cd - ch0) for both engines' tilings
    float gv[NC], av[NC], bv[NC];
#pragma unroll
    for (int j = 0; j < NC; ++j) {
      float pt = lo[j], ps = hi[j];
      if (bias) { pt += bias[ch0 + j]; ps += bias[Cd + ch0 + j]; }
      if (FAST && f16) {
        av[j] = tanh_ex2(pt);
        bv[j] = sigmoid_ex2(ps);
      } else {
        av[j] = tanh_f<FAST>(pt);
        bv[j] = sigmoid_f<FAST>(ps);
      }
      gv[j] = av[j] * bv[j];
    }
    long long o = row * Cd + ch0;
    store_ops<OpT, NC>(g + o, gv, f16);
    if (a_save) {
      store_ops<OpT, NC>(a_save + o, av, f16);
      store_ops<OpT, NC>(b_save + o, bv, f16);
    }
  }
};

// ---- 2. residual / skip: W_o output split (model/waveglow.py:45-46,104) -------------------------
template <typename OpT>
struct ResSkipEpi {
  static constexpr int kAux = 1;
  const float* res_src;  // [rows][Cr] fp32 layer input (nullptr when res_src_op is used)
  const OpT* res_src_op; // alternative residual source in operand type (ff training path)
  float* res_dst32;      // [rows][Cr] fp32 or nullptr
  OpT* res_dst_op;       // [rows][Cr] operand copy for the next layer or nullptr
  float* skip;           // [rows][Cs] fp32 cumulative skip
  const float* bias;     // nullptr or [nb]
  int Cr, Cs, cr_eff, first_layer, f16;
  const int* row_len;    // nullptr, or per-item lengths: the residual output is 0 at rows t >= row_len[b] (row = b * T + t)
  int T;
  template <int NC>
  __device__ __forceinline__ void load(long long row, int col0, float (&aux)[NC]) const {
    if (col0 < cr_eff) {
      long long o = row * Cr + col0;
      if (res_src) load_f32<NC>(res_src + o, aux);
      else load_ops<OpT, NC>(res_src_op + o, aux, f16);
    } else {
      int k = col0 - cr_eff;
      if (k < Cs && !first_layer) {
        load_f32<NC>(skip + row * Cs + k, aux);
      } else {
#pragma unroll
        for (int j = 0; j < NC; ++j) aux[j] = 0.f;
      }
    }
  }
  template <int NC>
  __device__ __forceinline__ void apply(long long row, int col0, const float (&v)[NC], const float (&aux)[NC]) const {
    float w[NC];
#pragma unroll
    for (int j = 0; j < NC; ++j) w[j] = v[j] + aux[j] + (bias ? bias[col0 + j] : 0.f);
    if (col0 < cr_eff) {
      if (row_len != nullptr) {
        const long long b = row / T;
        if (row - b * T >= __ldg(row_len + b)) {
#pragma unroll
          for (int j = 0; j < NC; ++j) w[j] = 0.f;
        }
      }
      long long o = row * Cr + col0;
      if (res_dst32) store_f32<NC>(res_dst32 + o, w);
      if (res_dst_op) store_ops<OpT, NC>(res_dst_op + o, w, f16);
    } else {
      int k = col0 - cr_eff;
      if (k >= Cs) return;
      store_f32<NC>(skip + row * Cs + k, w);
    }
  }
  template <int NC>
  __device__ __forceinline__ void op(long long row, int col0, const float (&v)[NC]) const {
    float aux[NC];
    load<NC>(row, col0, aux);
    apply<NC>(row, col0, v, aux);
  }
};

// ---- 3. gate backward: dpre = dg * d(tanh*sigmoid) ----------------------------------------------
template <typename OpT>
struct GateBwdEpi {
  static constexpr int kAux = 2;
  const OpT* a_save;  // tanh values
  const OpT* b_save;  // sigmoid values
  OpT* dpre;          // [rows][ld]: columns [0,Cd) tanh-half grads, [Cd,2Cd) sigmoid-half grads
  int Cd, ld, f16;
  template <int NC>
  __device__ __forceinline__ void load(long long row, int col0, float (&aux)[2 * NC]) const {
    if (col0 >= Cd) return;
    long long o = row * Cd + col0;
    load_ops<OpT, NC>(a_save + o, aux, f16);
    load_ops<OpT, NC>(b_save + o, aux + NC, f16);
  }
  template <int NC>
  __device__ __forceinline__ void apply(long long row, int col0, const float (&v)[NC], const float (&aux)[2 * NC]) const {
    if (col0 >= Cd) return;
    float dt[NC], ds[NC];
#pragma unroll
    for (int j = 0; j < NC; ++j) {
      float a = aux[j], b = aux[NC + j];
      dt[j] = v[j] * b * (1.f - a * a);
      ds[j] = v[j] * a * b * (1.f - b);
    }
    long long p = row * ld + col0;
    store_ops<OpT, NC>(dpre + p, dt, f16);
    store_ops<OpT, NC>(dpre + p + Cd, ds, f16);
  }
  template <int NC>
  __device__ __forceinline__ void op(long long row, int col0, const float (&v)[NC]) const {
    float aux[2 * NC];
    load<NC>(row, col0, aux);
    apply<NC>(row, col0, v, aux);
  }
};

// ---- 4. dx of the dilated conv + residual gradient ----------------------------------------------
template <typename OpT>
struct DxEpi {
  static constexpr int kAux = 1;
  const float* src;  // [rows][Cr] fp32 upstream residual gradient or nullptr (last layer)
  float* dst32;      // [rows][Cr]
  OpT* dst_op;       // operand copy or nullptr
  int Cr, f16;
  template <int NC>
  __device__ __forceinline__ void load(long long row, int col0, float (&aux)[NC]) const {
    if (src && col0 < Cr) {
      load_f32<NC>(src + row * Cr + col0, aux);
    } else {
#pragma unroll
      for (int j = 0; j < NC; ++j) aux[j] = 0.f;
    }
  }
  template <int NC>
  __device__ __forceinline__ void apply(long long row, int col0, const float (&v)[NC], const float (&aux)[NC]) const {
    if (col0 >= Cr) return;
    float w[NC];
#pragma unroll
    for (int j = 0; j < NC; ++j) w[j] = v[j] + aux[j];
    long long o = row * Cr + col0;
    store_f32<NC>(dst32 + o, w);
    if (dst_op) store_ops<OpT, NC>(dst_op + o, w, f16);
  }
  template <int NC>
  __device__ __forceinline__ void op(long long row, int col0, const float (&v)[NC]) const {
    float aux[NC];
    load<NC>(row, col0, aux);
    apply<NC>(row, col0, v, aux);
  }
};

// ---- 5. accumulate into an fp32 slab (conditioning gradient) ------------------------------------
struct AccumEpi {
  static constexpr int kAux = 1;
  float* dst;  // [rows][ld]
  int ld, n_valid, first;
  template <int NC>
  __device__ __forceinline__ void load(long long row, int col0, float (&aux)[NC]) const {
    if (!first && col0 < n_valid) {
      load_f32<NC>(dst + row * ld + col0, aux);
    } else {
#pragma unroll
      for (int j = 0; j < NC; ++j) aux[j] = 0.f;
    }
  }
  template <int NC>
  __device__ __forceinline__ void apply(long long row, int col0, const float (&v)[NC], const float (&aux)[NC]) const {
    if (col0 >= n_valid) return;
    float w[NC];
#pragma unroll
    for (int j = 0; j < NC; ++j) w[j] = v[j] + aux[j];
    store_f32<NC>(dst + row * ld + col0, w);
  }
  template <int NC>
  __device__ __forceinline__ void op(long long row, int col0, const float (&v)[NC]) const {
    float aux[NC];
    load<NC>(row, col0, aux);
    apply<NC>(row, col0, v, aux);
  }
};

// ---- 6. plain fp32 store (self tests) -----------------------------------------------------------
struct StoreEpi {
  static constexpr int kAux = 1;
  float* dst;  // [rows][ld]
  int ld, n_valid;
  const float* bias;  // nullptr or [n_valid]
  template <int NC>
  __device__ __forceinline__ void load(long long, int, float (&aux)[NC]) const {
#pragma unroll
    for (int j = 0; j < NC; ++j) aux[j] = 0.f;
  }
  template <int NC>
  __device__ __forceinline__ void apply(long long row, int col0, const float (&v)[NC], const float (&)[NC]) const {
    op<NC>(row, col0, v);
  }
  template <int NC>
  __device__ __forceinline__ void op(long long row, int col0, const float (&v)[NC]) const {
    if (col0 >= n_valid) return;
    float w[NC];
#pragma unroll
    for (int j = 0; j < NC; ++j) w[j] = v[j] + (bias ? bias[col0 + j] : 0.f);
    store_f32<NC>(dst + row * ld + col0, w);
  }
};

}  // namespace cmwg
