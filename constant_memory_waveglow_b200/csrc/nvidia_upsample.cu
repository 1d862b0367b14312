// Conditioning of NVIDIA's WaveGlow (NVIDIA/waveglow glow.py): a dense ConvTranspose1d(C, C, taps * hop, stride = hop)
// with bias at the sample rate, then unfolded by n_group into C * n_group channels at the squeezed rate, as ONE tcgen05
// GEMM (engine_tc.cuh) whose epilogue writes the WN's 16-bit conditioning slab directly.
//
//   up[b, o, hop q + r] = bias[o] + sum_{j < taps} sum_i W[i, o, r + hop j] * mel[b, i, q - j]     (mel = 0 outside [0, F))
//   slab[b][t][c] = up[b, c / n_group, n_group t + c % n_group]      (channel c of squeezed step t; the WN's ycl layout)
//
// GEMM: row q = mel frame; K = taps x C, k = j C + i (the operand row q holds mel frames q, q-1, .., q-taps+1 side by
// side, zero outside [0, F), so K has no padding beyond the next multiple of 64: 320 for the published 80 x 4);
// column n = (r / n_group) * (C n_group) + o * n_group + r % n_group.  Row q x columns [0, hop C) is then exactly the
// hop / n_group squeezed steps (hop / n_group) q .. (hop / n_group)(q + 1) - 1 of the slab, C n_group channels each:
// the output of the GEMM, read as [B][frames][hop C], IS the slab [B][T][C n_group] when T fills whole frames.
#include "engine_tc.cuh"
#include "epilogues_tc.cuh"

namespace cmwg {

// out = rn16(acc + bias[o]) with o = (n % (C n_group)) / n_group
struct UpsampleSlabTcEpi {
  static constexpr bool kPaired = false, kOutF32 = false;
  static constexpr int kOut = 1, kIn = 0, kOutBufs = 2, kColGroups = 4;
  const float* bias;
  int width;    // C * n_group: slab channels
  int n_group;
  int f16;
  __device__ __forceinline__ int out_col(int, int c0) const { return c0; }
  __device__ __forceinline__ int in_col(int, int c0) const { return c0; }
  __device__ __forceinline__ void compute(int col0, float (&v)[16], uint32_t (&o)[1][8]) const {
    const int c0 = col0 % width;  // 16 columns never straddle a squeezed step: width is a multiple of 64
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] += __ldg(bias + (c0 + j) / n_group);
    if (f16) {
#pragma unroll
      for (int j = 0; j < 16; j += 2) o[0][j >> 1] = pack2(v[j], v[j + 1], 1);
    } else {
#pragma unroll
      for (int j = 0; j < 16; j += 2) o[0][j >> 1] = pack2(v[j], v[j + 1], 0);
    }
  }
};

// B operand [hop C][Kp]: wp[n][j C + i] = W[i, o(n), r(n) + hop j]; k >= taps C is zero
__global__ void __launch_bounds__(256) nv_ups_pack_kernel(const float* __restrict__ w, int C, int hop, int taps,
                                                          int n_group, int Kp, uint16_t* __restrict__ wp, int f16) {
  const int n = blockIdx.x;
  const int width = C * n_group;
  const int r = (n / width) * n_group + n % n_group, o = (n % width) / n_group;
  const int L = taps * hop;
  for (int k = threadIdx.x; k < Kp; k += 256) {
    float val = 0.f;
    if (k < taps * C) {
      const int j = k / C, i = k % C;
      val = w[((long long)i * C + o) * L + r + hop * j];
    }
    wp[(long long)n * Kp + k] = f32_to_op16(val, f16);
  }
}

// A operand [B][Fq][Kp]: a[b][q][j C + i] = mel[b, i, q - j] (0 outside [0, F) and for k >= taps C)
__global__ void __launch_bounds__(256) nv_ups_operand_kernel(const float* __restrict__ mel, long long bs, long long cs,
                                                             int C, int F, int Fq, int taps, int Kp,
                                                             uint16_t* __restrict__ a, int f16) {
  const int q = blockIdx.x, b = blockIdx.y;
  for (int k = threadIdx.x; k < Kp; k += 256) {
    float val = 0.f;
    if (k < taps * C) {
      const int j = k / C, i = k % C, f = q - j;
      if (f >= 0 && f < F) val = mel[b * bs + i * cs + f];
    }
    a[((long long)b * Fq + q) * Kp + k] = f32_to_op16(val, f16);
  }
}

struct NvUpsDims {
  int Kp, N, width, rows_per_frame, Fq;
  bool direct;   // the slab holds whole frames: the GEMM stores into it; otherwise into the workspace, then a 2-D copy
};

static int nv_ups_dims(int C, int hop, int taps, int n_group, int T, NvUpsDims* d) {
  CMWG_REQUIRE(C >= 1 && hop >= 1 && taps >= 1 && n_group >= 1 && T >= 0, "nvidia upsample: bad dims");
  CMWG_REQUIRE(hop % n_group == 0, "nvidia upsample: n_group %d does not divide the hop %d", n_group, hop);
  if ((C * n_group) % 64 != 0) {
    set_error("nvidia upsample: C * n_group = %d is not a multiple of 64 (the 16-bit WN slab's channel tile)",
              C * n_group);
    return CMWG_ERR_UNSUPPORTED;
  }
  d->Kp = round_up(taps * C, TC_BK);
  d->width = C * n_group;
  d->N = hop * C;
  d->rows_per_frame = hop / n_group;
  d->Fq = ceil_div(T, d->rows_per_frame);
  d->direct = (long long)d->Fq * d->rows_per_frame == T;
  return CMWG_OK;
}

}  // namespace cmwg

using namespace cmwg;

extern "C" {

size_t cmwg_nvidia_upsample_packed_bytes(int C, int hop, int taps) {
  if (C < 1 || hop < 1 || taps < 1) return 0;
  return (size_t)hop * C * round_up(taps * C, TC_BK) * sizeof(uint16_t);
}

int cmwg_nvidia_upsample_pack(const float* w, int C, int hop, int taps, int n_group, int precision, void* packed,
                              void* stream) {
  NvUpsDims d;
  CMWG_PROPAGATE(nv_ups_dims(C, hop, taps, n_group, 0, &d));
  CMWG_REQUIRE(w && packed, "cmwg_nvidia_upsample_pack: null argument");
  CMWG_REQUIRE(precision == CMWG_PREC_FP16 || precision == CMWG_PREC_BF16,
               "cmwg_nvidia_upsample_pack: precision %d is not a 16-bit operand type", precision);
  nv_ups_pack_kernel<<<d.N, 256, 0, (cudaStream_t)stream>>>(w, C, hop, taps, n_group, d.Kp, (uint16_t*)packed,
                                                           precision == CMWG_PREC_FP16);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

size_t cmwg_nvidia_upsample_workspace_bytes(int B, int T, int C, int hop, int taps, int n_group) {
  NvUpsDims d;
  if (B < 0 || nv_ups_dims(C, hop, taps, n_group, T, &d) != CMWG_OK) return 0;
  size_t bytes = align_up((size_t)B * d.Fq * d.Kp * sizeof(uint16_t), 1024);
  if (!d.direct) bytes += (size_t)B * d.Fq * d.N * sizeof(uint16_t);
  return bytes + 1024;
}

int cmwg_nvidia_upsample_slab(const void* packed, const float* bias, const float* mel, long long mel_bstride,
                              long long mel_cstride, int B, int C, int F, int hop, int taps, int n_group, int T,
                              int precision, void* slab, void* workspace, void* stream) {
  NvUpsDims d;
  CMWG_PROPAGATE(nv_ups_dims(C, hop, taps, n_group, T, &d));
  CMWG_REQUIRE(packed && bias && mel && slab && workspace, "cmwg_nvidia_upsample_slab: null argument");
  CMWG_REQUIRE(B >= 0 && F >= 1, "cmwg_nvidia_upsample_slab: bad batch %d / frames %d", B, F);
  CMWG_REQUIRE(precision == CMWG_PREC_FP16 || precision == CMWG_PREC_BF16,
               "cmwg_nvidia_upsample_slab: precision %d is not a 16-bit operand type", precision);
  if (B == 0 || T == 0) return CMWG_OK;
  const int f16 = precision == CMWG_PREC_FP16;
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* ws = reinterpret_cast<uint8_t*>(align_up(reinterpret_cast<uintptr_t>(workspace), 1024));
  uint16_t* a = reinterpret_cast<uint16_t*>(ws);
  void* out = d.direct ? slab : ws + align_up((size_t)B * d.Fq * d.Kp * sizeof(uint16_t), 1024);

  nv_ups_operand_kernel<<<dim3(d.Fq, B), 256, 0, st>>>(mel, mel_bstride, mel_cstride, C, F, d.Fq, taps, d.Kp, a, f16);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();

  GemmDesc g;
  memset(&g, 0, sizeof(g));
  g.nseg = 1;
  g.seg[0].a = a; g.seg[0].lda = d.Kp; g.seg[0].K = d.Kp;
  g.w = packed; g.ldw = d.Kp; g.N = d.N; g.n_rows_w = d.N;
  g.B = B; g.T = d.Fq; g.bn = 256; g.is_fp16 = f16;
  g.tag = CMWG_KCLASS_GATE;   // the conditioning term of the gate GEMMs, computed once per call
  TcIo io;
  memset(&io, 0, sizeof(io));
  io.out[0] = TcStream{out, d.N, d.N, 0};
  UpsampleSlabTcEpi epi{bias, d.width, n_group, f16};
  CMWG_PROPAGATE(tc_gemm_launch<UpsampleSlabTcEpi>(g, io, epi, st));
  if (!d.direct) {  // keep the first T squeezed steps of every item
    const size_t row = (size_t)d.width * sizeof(uint16_t);
    CMWG_CHECK_CUDA(cudaMemcpy2DAsync(slab, (size_t)T * row, out, (size_t)d.Fq * d.rows_per_frame * row, (size_t)T * row,
                                      B, cudaMemcpyDeviceToDevice, st));
  }
  return CMWG_OK;
}

}  // extern "C"
