// Shared helpers for the cmwg_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/cmwg_b200.h"

namespace cmwg {

// ------------------------------------------------------------------------------------------
// error plumbing: no exceptions cross the C ABI; every entry point returns an int and leaves a
// message retrievable through cmwg_last_error().
// ------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);

#define CMWG_CHECK_CUDA(expr)                                                                \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      ::cmwg::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #expr,                   \
                        cudaGetErrorString(_e));                                             \
      return CMWG_ERR_CUDA;                                                                  \
    }                                                                                        \
  } while (0)

#define CMWG_REQUIRE(cond, ...)                                                              \
  do {                                                                                       \
    if (!(cond)) {                                                                           \
      ::cmwg::set_error(__VA_ARGS__);                                                        \
      return CMWG_ERR_ARG;                                                                   \
    }                                                                                        \
  } while (0)

#define CMWG_PROPAGATE(expr)                                                                 \
  do {                                                                                       \
    int _r = (expr);                                                                         \
    if (_r != CMWG_OK) return _r;                                                            \
  } while (0)

#define CMWG_LAUNCH_CHECK() CMWG_CHECK_CUDA(cudaGetLastError())

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline long long ceil_div_ll(long long a, long long b) { return (a + b - 1) / b; }
static inline int round_up(int a, int b) { return ceil_div(a, b) * b; }
static inline size_t align_up(size_t a, size_t b) { return (a + b - 1) / b * b; }

int num_sms();

// optional per-kernel-class event timing (bench.py's roofline leg); no-ops unless enabled
void prof_begin(cudaStream_t st, int cls);
void prof_end(cudaStream_t st);
struct ProfScope {
  cudaStream_t st;
  ProfScope(cudaStream_t s, int cls) : st(s) { prof_begin(s, cls); }
  ~ProfScope() { prof_end(st); }
};

// ------------------------------------------------------------------------------------------
// Programmatic dependent launch (PDL): a kernel launched through launch_pdl() may start -- be scheduled on free
// SMs, allocate TMEM, initialise barriers, prefetch tensor maps -- while its predecessor in the stream is still
// running; it must execute pdl_wait() before it touches global memory (the wait returns once the predecessor
// grid has completed and flushed).  pdl_trigger() at the top of a kernel lets ITS successor start equally early.
// The short per-line kernels of WaveFlow's row-recurrent inverse and the launch gaps of the synthesis chains are
// what this buys back.  CMWG_PDL=0 falls back to plain stream-ordered launches.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
bool pdl_enabled();

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// kernel launch counter (bench.py reports it as gpu_launches)
extern unsigned long long g_launch_count;
#define CMWG_COUNT_LAUNCH() (++::cmwg::g_launch_count)

// ------------------------------------------------------------------------------------------
// operand element types: the WN GEMM operands are stored either as fp32 (exact CUDA-core engine)
// or as 16-bit (bf16 / fp16) for the tcgen05 engine.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint16_t f32_to_op16(float v, int is_fp16) {
  if (is_fp16) {
    // saturate instead of producing inf
    v = fminf(fmaxf(v, -65504.f), 65504.f);
    return __half_as_ushort(__float2half_rn(v));
  }
  return __bfloat16_as_ushort(__float2bfloat16_rn(v));
}
__device__ __forceinline__ float op16_to_f32(uint16_t u, int is_fp16) {
  if (is_fp16) return __half2float(__ushort_as_half(u));
  return __bfloat162float(__ushort_as_bfloat16(u));
}

template <typename T> struct OpTraits;
template <> struct OpTraits<float> {
  static constexpr bool is16 = false;
  __device__ __forceinline__ static float load(const float* p, int) { return *p; }
  __device__ __forceinline__ static void store(float* p, float v, int) { *p = v; }
};
template <> struct OpTraits<uint16_t> {
  static constexpr bool is16 = true;
  __device__ __forceinline__ static float load(const uint16_t* p, int f16) { return op16_to_f32(*p, f16); }
  __device__ __forceinline__ static void store(uint16_t* p, float v, int f16) { *p = f32_to_op16(v, f16); }
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// sum of v over the CTA (blockDim.x <= 1024) in a fixed order; red holds 32 floats of shared memory
__device__ __forceinline__ float block_sum_1024(float v, float* red) {
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

// accurate (fp32 mode) and fast (tensor-core modes) gate non-linearities
template <bool FAST> __device__ __forceinline__ float tanh_f(float x) {
  if (FAST) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
  }
  return tanhf(x);
}
template <bool FAST> __device__ __forceinline__ float sigmoid_f(float x) {
  if (FAST) return fmaf(0.5f, tanh_f<true>(0.5f * x), 0.5f);
  return 1.f / (1.f + expf(-x));
}
// MUFU.EX2 + MUFU.RCP forms: ~1e-7 absolute error (tanh.approx is ~5e-4), used with fp16 operands
// whose 11-bit mantissa would otherwise be wasted on the gate approximation
__device__ __forceinline__ float tanh_ex2(float x) { return 1.f - __fdividef(2.f, 1.f + __expf(2.f * x)); }
__device__ __forceinline__ float sigmoid_ex2(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }
// tanh(x), sigmoid(y) and their product with ONE reciprocal:  E1 = e^(2x), E2 = e^(-y), r = 1 / ((E1 + 1)(1 + E2));
//   tanh = (E1 - 1)(1 + E2) r,  sigmoid = (E1 + 1) r,  tanh * sigmoid = (E1 - 1) r.
// x is clamped above at 15 (tanh = 1 to fp32 precision beyond 9.1) and y below at -30 so that the product stays finite.
template <bool WANT_AB>
__device__ __forceinline__ void gate_ex2(float x, float y, float& a, float& b, float& g) {
  float e1, e2, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(fminf(x, 15.f) * 2.885390082f));   // 2 log2(e)
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e2) : "f"(fmaxf(y, -30.f) * -1.442695041f));
  const float p = e1 + 1.f, q = 1.f + e2, m = e1 - 1.f;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(p * q));
  g = m * r;
  if (WANT_AB) {
    b = p * r;
    a = m * q * r;
  }
}

}  // namespace cmwg
