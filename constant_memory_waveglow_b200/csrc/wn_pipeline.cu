// WN transform: forward, backward, weight packing.  Orchestrates the GEMM engines (engine_tc.cuh /
// engine_ff.cuh) and the CUDA-core kernels of wn_kernels.cuh; exported through the C ABI.
//
// Per NonCausalLayer i (model/waveglow.py:41-46), forward:
//   gate GEMM   pre[row][2Cd] = sum_tap h_i[row + (tap-c)*2^i] W_tap^T  +  ycond[row] V_i^T
//               (the conditioning 1x1 conv V is folded in as extra K rows, so its (B, 2*Cd*depth, T)
//               output -- 786 MB per flow at the LJ config -- never exists), epilogue = fused_gate
//   res/skip GEMM  ro = g W_o^T ; epilogue: h_{i+1} = h_i + ro[:, :Cr] (fp32 stream + operand copy),
//               skip += ro[:, Cr:] (fp32)
// backward (reverse layer order), given d(end output):
//   dgate GEMM  dg = [dh_{i+1} | dskip] W_o ; epilogue: dpre = dg * d(tanh*sigmoid)
//   wgrad GEMMs dW_o, dW (per tap), dV_i: MN-major reads of the same slabs, split-K over time
//   dcond GEMM  dycond += dpre V_i
//   dx GEMM     dh_i = dh_{i+1} + sum_tap dpre[row - (tap-c)*2^i] W_tap
#include "engine_ff.cuh"
#include "engine_tc.cuh"
#include "engine_mega.cuh"
#include "epilogues.cuh"
#include "epilogues_tc.cuh"
#include "wn_kernels.cuh"

namespace cmwg {

template <typename OpT> struct EngineSel;
template <> struct EngineSel<float> {
  static constexpr bool kTc = false;
  template <bool PAIRED, class Epi>
  static int gemm(const GemmDesc& d, const Epi& e, cudaStream_t st) { return ff_gemm_launch<Epi, PAIRED>(d, e, st); }
};
template <> struct EngineSel<uint16_t> {
  static constexpr bool kTc = true;
  template <bool PAIRED, class Epi>
  static int gemm(const GemmDesc&, const Epi&, cudaStream_t) {  // the tc engine has its own functors (epilogues_tc.cuh)
    set_error("internal: FFMA epilogue functor routed to the tcgen05 engine");
    return CMWG_ERR_ARG;
  }
};

static inline TcStream op_stream(const void* p, int ld) { return TcStream{p, ld, ld, 0}; }
static inline TcStream f32_stream(const void* p, int ld) { return TcStream{p, ld, ld, 1}; }

static inline int pick_bn(int N) { return N >= 256 ? 256 : 128; }

static inline const uint8_t* cu8(const void* p) { return reinterpret_cast<const uint8_t*>(p); }
static inline uint8_t* u8(void* p) { return reinterpret_cast<uint8_t*>(p); }

// ------------------------------------------------------------------------------------------------
// pack
// ------------------------------------------------------------------------------------------------
static int wn_pack_impl(const WnDims& d, const cmwg_wn_params* prm, void* packed, cudaStream_t st) {
  PackedLayout L = make_packed_layout(d);
  uint8_t* base = u8(packed);
  WeffTable tb;
  int n = 0, rows = 0;
  auto add = [&](const cmwg_conv_param& c, size_t w_off, size_t n_off, int O, int Lr) {
    WeffEntry& e = tb.e[n++];
    e.g = c.g; e.v = c.v;
    e.w = reinterpret_cast<float*>(base + w_off);
    e.inv_norm = c.g ? reinterpret_cast<float*>(base + n_off) : nullptr;
    e.O = O; e.L = Lr; e.row_begin = rows;
    rows += O;
  };
  CMWG_REQUIRE(prm->V.v && prm->start.v && prm->end.v, "cmwg_wn_pack: missing V/start/end weights");
  add(prm->V, L.wV, L.nV, 2 * d.Cd * d.depth, d.aux);
  add(prm->start, L.wStart, L.nStart, d.Cr, d.cin);
  add(prm->end, L.wEnd, 0, 2 * d.cin, d.Cs);
  for (int i = 0; i < d.depth; ++i) {
    CMWG_REQUIRE(prm->W[i].v && prm->W_o[i].v, "cmwg_wn_pack: missing layer %d weights", i);
    add(prm->W[i], L.wW[i], L.nW[i], 2 * d.Cd, d.Cr * d.R);
    add(prm->W_o[i], L.wWo[i], L.nWo[i], d.nb(i), d.Cd);
  }
  tb.n = n;
  if (2 * d.cin < 16)   // zero rows behind the `end` weights: the fused epilogue of the task kernel reads 8 or 16 rows
    CMWG_CHECK_CUDA(cudaMemsetAsync(base + L.wEnd + (size_t)2 * d.cin * d.Cs * 4, 0, (size_t)(16 - 2 * d.cin) * d.Cs * 4, st));
  weight_eff_kernel<<<rows, 128, 0, st>>>(tb);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();

  PackParams pp;
  pp.d = d;
  pp.wV = reinterpret_cast<const float*>(base + L.wV);
  pp.is_fp16 = d.prec == CMWG_PREC_FP16;
  for (int i = 0; i < d.depth; ++i) {
    pp.wW[i] = reinterpret_cast<const float*>(base + L.wW[i]);
    pp.wWo[i] = reinterpret_cast<const float*>(base + L.wWo[i]);
    pp.PA[i] = base + L.PA[i]; pp.PB[i] = base + L.PB[i]; pp.Q1[i] = base + L.Q1[i];
    pp.Q2[i] = base + L.Q2[i];
  }
  pp.QV = base + L.QV[0];
  pp.PS = base + L.PS;
  long long biggest = (long long)d.npadA * d.KA;
  long long q2 = (long long)d.Cr * d.ldQ2;
  if (q2 > biggest) biggest = q2;
  int gx = (int)std::min<long long>(ceil_div_ll(biggest, 256 * 4), 1024);
  dim3 grid(gx, d.depth, d.tc ? 6 : 5);
  const char* pse = getenv("CMWG_PACK_SCALAR");   // =1: the one-element-per-thread kernel (tests compare the two)
  const bool pack_scalar = pse && pse[0] == '1';
  if (d.tc && !pack_scalar) {
    // vector form: the largest matrix (PA) has npadA * (Crp + auxp) / 8 work items
    const long long items = (long long)d.npadA * ((d.Crp + d.auxp) / 8);
    grid.x = (unsigned)std::max<long long>(1, std::min<long long>(ceil_div_ll(items, 256), 1024));
    pack_operands16_kernel<<<grid, 256, 0, st>>>(pp);
  } else if (d.tc) {
    pack_operands_kernel<uint16_t><<<grid, 256, 0, st>>>(pp);
  } else {
    pack_operands_kernel<float><<<grid, 256, 0, st>>>(pp);
  }
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();

  if (fold0_shapes_ok(d)) {   // layer 0 with the start conv folded in (used by the task kernel's forward)
    Fold0Params fp;
    fp.d = d;
    fp.wV = reinterpret_cast<const float*>(base + L.wV);
    fp.wW0 = reinterpret_cast<const float*>(base + L.wW[0]);
    fp.wWo0 = reinterpret_cast<const float*>(base + L.wWo[0]);
    fp.wStart = reinterpret_cast<const float*>(base + L.wStart);
    fp.PA0f = reinterpret_cast<uint16_t*>(base + L.PA0f);
    fp.PB0f = reinterpret_cast<uint16_t*>(base + L.PB0f);
    fp.is_fp16 = d.prec == CMWG_PREC_FP16;
    const long long n = (long long)d.npadA * d.auxp + (long long)d.Cr * (d.Cdp + d.kb);
    const int nb_dot = (int)ceil_div_ll((long long)d.npadA * d.R * d.cin * 32, 256);
    pack_fold0_kernel<<<(int)ceil_div_ll(n, 256) + nb_dot, 256, 0, st>>>(fp);
    CMWG_COUNT_LAUNCH();
    CMWG_LAUNCH_CHECK();
  }

  if (foldend_shapes_ok(d)) {   // dgate weights with the `end` conv folded in (used by the task kernel's backward chain)
    FoldEndParams ep;
    ep.d = d;
    ep.wEnd = reinterpret_cast<const float*>(base + L.wEnd);
    ep.is_fp16 = d.prec == CMWG_PREC_FP16;
    for (int i = 0; i < d.depth; ++i) {
      ep.wWo[i] = reinterpret_cast<const float*>(base + L.wWo[i]);
      ep.Q1f[i] = reinterpret_cast<uint16_t*>(base + L.Q1f[i]);
    }
    const int nb_t = ceil_div(d.Cd * (k1f(d, 0) / 16), 256);     // layer 0 has the widest matrix (depth >= 2) or the only one
    pack_foldend_kernel<<<dim3(nb_t + ceil_div(d.Cd, 32), d.depth), 256, 0, st>>>(ep);
    CMWG_COUNT_LAUNCH();
    CMWG_LAUNCH_CHECK();
  }

  if (d.bias) {
    BiasPackParams bp;
    bp.d = d;
    CMWG_REQUIRE(prm->V.bias && prm->start.bias && prm->end.bias, "cmwg_wn_pack: has_bias set but bias pointers missing");
    bp.bV = prm->V.bias; bp.bStart = prm->start.bias; bp.bEnd = prm->end.bias;
    bp.biasStart = reinterpret_cast<float*>(base + L.biasStart);
    bp.biasEnd = reinterpret_cast<float*>(base + L.biasEnd);
    bp.biasS = reinterpret_cast<float*>(base + L.biasS);
    for (int i = 0; i < d.depth; ++i) {
      CMWG_REQUIRE(prm->W[i].bias && prm->W_o[i].bias, "cmwg_wn_pack: layer %d bias missing", i);
      bp.bW[i] = prm->W[i].bias; bp.bWo[i] = prm->W_o[i].bias;
      bp.biasA[i] = reinterpret_cast<float*>(base + L.biasA[i]);
      bp.biasB[i] = reinterpret_cast<float*>(base + L.biasB[i]);
    }
    pack_bias_kernel<<<dim3(4, d.depth), 256, 0, st>>>(bp);
    CMWG_COUNT_LAUNCH();
    CMWG_LAUNCH_CHECK();
  }
  return CMWG_OK;
}

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
// Line window of the row-recurrent inverse of the 2-D WN (model/waveflow.py:53-67,137-151,243-258): only lines
// [h0, h0 + nh) are computed; `state` holds every layer's input slab for ALL lines (the reference's rolling
// per-layer buffers), so a tap reaching up to line h - 2*h_dilation finds what earlier calls left there.
struct LineWin {
  void* state = nullptr;
  int h0 = 0, nh = 0;  // nh = 0: all lines
};

static inline size_t line_state_slab_bytes(const WnDims& d, int B, int T) {
  return align_up((size_t)B * d.H * T * d.Cr * d.opsize, 1024);
}

// Per-item lengths of a padded batch (cmwg_wn_forward_varlen): item b has valid rows [0, len[b]).  `host` plans the task
// kernel's list (only row tiles that hold valid rows); `dev` (the same values, on the device) drives the masks that keep every
// layer input zero from row len[b] on -- what the TMA zero fill gives a call of length len[b].
struct VarLen {
  const int* host = nullptr;
  const int* dev = nullptr;
  bool on() const { return dev != nullptr; }
};

// row-tile table of the task kernel for per-item lengths (MegaParams::rt_tab), in the workspace behind the layouts
static inline size_t varlen_tab_offset(const WnDims& d, int B, int T) {
  FwdLayout FL;
  make_fwd_layout(d, B, T, &FL);
  BwdLayout BL;
  make_bwd_layout(d, B, T, &BL);
  return align_up(FL.ws_total > BL.total ? FL.ws_total : BL.total, 1024);
}
static inline int varlen_row_tiles(const int* len, int B) {
  int rt = 0;
  for (int b = 0; b < B; ++b) rt += ceil_div(len[b], 2 * TC_BM);
  return rt;
}


// ------------------------------------------------------------------------------------------------
// single-kernel forward (engine_mega.cuh): every gate / residual / skip GEMM tile of the WN as one task list
// ------------------------------------------------------------------------------------------------
static long long* g_mega_clk = nullptr;
static bool mega_enabled() {  // read at every call: tests flip CMWG_MEGA inside one process
  const char* v = getenv("CMWG_MEGA");
  return !(v && v[0] == '0');
}

// residual (forward) / dgate (backward) tiles trail their gate / dx tiles by `lag` row-tile slots; lag <= RT - 2 keeps the
// list in dependency order (tests/test_host.py::test_task_lists_are_in_dependency_order)
static inline int mega_fwd_lag(int RT) {
  static const int lag_env = [] { const char* v = getenv("CMWG_MEGA_LAG"); return v ? atoi(v) : 64; }();
  return std::max(0, std::min(lag_env, RT - 2));
}
static inline int mega_bwd_lag(int RT) {
  static const int lag_env = [] { const char* v = getenv("CMWG_MEGA_LAG_BWD"); return v ? atoi(v) : 96; }();
  return std::max(0, std::min(lag_env, RT - 2));
}

static inline int mega_dual() {  // CMWG_MEGA_DUAL=0: one TMA producer thread for both operands (the round-1 arrangement)
  static const int v = [] { const char* e = getenv("CMWG_MEGA_DUAL"); return (e && e[0] == '0') ? 0 : 1; }();
  return v;
}

// CMWG_GATE_MIX=1: every second gate value takes its sigmoid exponential from the FMA pipe (exp2_fma) instead of MUFU.EX2.
// Measured: the gate epilogue gets 11 % shorter (3559 -> 3177 cycles per tile) and the kernel does not get faster (0.504 ms
// either way: the residual tiles' epilogue and the operand feed bound it), so it stays off.
static inline int gate_mix() {
  static const int v = [] { const char* e = getenv("CMWG_GATE_MIX"); return (e && e[0] == '1') ? 1 : 0; }();
  return v;
}

// Residual stream of the tcgen05 engine (forward) and its gradient (backward): (hi, lo) pair of 16-bit slabs, or the operand
// slab alone (AddTcEpi: fp16 operands only -- bf16's 8 mantissa bits need the pair).  CMWG_RES_LO=1 keeps the pair with fp16
// too (read at every call).
static inline bool fwd_res_lo(const WnDims& d) {
  if (d.prec != CMWG_PREC_FP16) return true;
  const char* e = getenv("CMWG_RES_LO");
  return e && e[0] == '1';
}

// Layer 0 without the start conv (PackedLayout::PA0f / PB0f) in the task kernel's forward -- both variants: the first pass
// and the recompute of the reversible backward must produce the SAME log_s / t, or the input reconstructed from the output
// (efficient_modules.py:127-136) drifts by the difference, flow after flow.  h_0 is then never materialised; the one
// consumer besides layer 0 itself, the weight gradient of layer 0's dilated conv, goes through the fold as well
// (fold0_dw_kernel).  Needs the single-stream residual (the first residual tile has nothing to add).
// CMWG_FOLD0=0 turns it off (read at every call -- forward and backward of one step must see the same value).
static inline bool fold0_enabled(const WnDims& d) {
  if (!fold0_shapes_ok(d) || fwd_res_lo(d)) return false;
  const char* e = getenv("CMWG_FOLD0");
  return !(e && e[0] == '0');
}

// `end` conv folded into the dgate tiles of the backward task kernel (PackedLayout::Q1f).  CMWG_FOLD_END=0 turns it off.
static inline bool foldend_enabled(const WnDims& d) {
  if (!foldend_shapes_ok(d)) return false;
  const char* e = getenv("CMWG_FOLD_END");
  return !(e && e[0] == '0');
}

static inline bool mega_shapes_ok(const WnDims& d, int B, int T);
// The backward will run the single-kernel chain / batch all weight-gradient GEMMs / fold the `end` conv completely
// (wn_backward_impl); the saving forward asks the last one to know whether anything will read the fp32 skip sum.
static inline bool bwd_fused_chain(const WnDims& d, int B, int T) {
  const char* e = getenv("CMWG_MEGA_BWD");
  return d.tc && mega_enabled() && mega_shapes_ok(d, B, T) && d.Cd == 256 && !(e && e[0] == '0');
}
static inline bool bwd_wgrad_batched(const WnDims& d, int B, int T) {
  const char* e = getenv("CMWG_WGRAD_BATCH");
  return bwd_fused_chain(d, B, T) && d.depth * (d.R + 3) <= TC_MAX_WG && !(e && e[0] == '0');
}
static inline bool bwd_foldend_full(const WnDims& d, int B, int T) {
  const char* e = getenv("CMWG_FOLD_END_W");
  return bwd_wgrad_batched(d, B, T) && foldend_enabled(d) && !(e && e[0] == '0');
}

static inline bool mega_shapes_ok(const WnDims& d, int B, int T) {
  return d.tc && d.H == 1 && !d.bias && d.depth >= 1 && d.depth <= MEGA_D && d.Cr == 256 && d.Cs == 256 &&
         d.Cd % 128 == 0 && d.bn_gate == 256 && (((d.radix - 1) / 2) << (d.depth - 1)) <= 2 * TC_BM && d.radix <= 7 &&
         B >= 1 && T >= 1;
}

template <bool SAVE, bool VARLEN = false>
static int mega_launch(const MegaParams& p, cudaStream_t st) {
  auto kern = wn_fwd_mega_kernel<SAVE, VARLEN>;
  constexpr size_t smem = mega_smem_bytes<SAVE>();
  static_assert(smem <= TC_SMEM_LIMIT, "shared memory budget exceeded");
  static bool attr_set = false;
  if (!attr_set) {
    CMWG_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set = true;
  }
  const int pairs = std::min(p.total_tasks, num_sms() / 2);
  ProfScope prof(st, CMWG_KCLASS_FWDFUSED);
  void* args[1] = {(void*)&p};
  CMWG_PROPAGATE(tc_launch_pairs_coresident((const void*)kern, smem, pairs, args, st, MEGA_THREADS));
  CMWG_COUNT_LAUNCH();
  return CMWG_OK;
}

// hin(i) / hlo(i): (hi, lo) slabs of layer i's input; gop(i), sb(i): gate output and saved sigmoid
static inline bool mega_end_fused(const WnDims& d) {  // CMWG_MEGA_END=0: separate end conv kernel (read at every call: tests flip it)
  const char* e = getenv("CMWG_MEGA_END");
  return !(e && e[0] == '0') && 2 * d.cin <= MEGA_END_MAXC && !d.bias && d.Cs == MEGA_BN;
}

// tab[rt] = (item, tile within the item, tiles of the item) for the RT row tiles of per-item lengths len (clamped to [1, T]:
// a device copy that disagrees with the planning copy must not index outside the slabs)
static __global__ void varlen_tiles_kernel(const int* __restrict__ len, int B, int T, int RT, int4* __restrict__ tab) {
  const int rt = blockIdx.x * blockDim.x + threadIdx.x;
  if (rt >= RT) return;
  int start = 0;
  for (int b = 0; b < B; ++b) {
    const int n = (min(max(len[b], 1), T) + 2 * TC_BM - 1) / (2 * TC_BM);
    if (rt < start + n || b == B - 1) {
      const int tb = min(rt - start, n - 1);
      tab[rt] = make_int4(b, tb, n, 0);
      return;
    }
    start += n;
  }
}

// rows [end, min(T, end + rows)) of item blockIdx.x, end = its last row tile's end, zeroed in slab blockIdx.y (a or b)
static __global__ void varlen_zero_tail_kernel(const int* __restrict__ len, int T, int rows, int C, uint16_t* a, uint16_t* b) {
  const int item = blockIdx.x;
  const int end = (min(max(len[item], 1), T) + 2 * TC_BM - 1) / (2 * TC_BM) * (2 * TC_BM);
  const int n = min(T, end + rows) - end;
  if (n <= 0) return;
  uint16_t* slab = blockIdx.y ? b : a;
  uint4* p = reinterpret_cast<uint4*>(slab + ((size_t)item * T + end) * C);
  const long long nv = (long long)n * C / 8;
  for (long long i = threadIdx.x; i < nv; i += blockDim.x) p[i] = make_uint4(0u, 0u, 0u, 0u);
}

static int wn_forward_mega(const WnDims& d, const PackedLayout& PL, const FwdLayout& FL, const uint8_t* pk, uint8_t* ws,
                           const void* ycl, int B, int T, bool save, bool fold0, int f16, void* const* hin, void* const* hlo,
                           void* const* gop, void* const* sb, float* skip32, float* lst, cudaStream_t st,
                           const VarLen& vl = VarLen()) {
  MegaParams p;
  memset(&p, 0, sizeof(p));
  const bool res_lo = fwd_res_lo(d);
  p.res_lo = res_lo ? 1 : 0;
  for (int i = 0; i < d.depth; ++i) {
    CMWG_PROPAGATE(get_slab_map(&p.hin_op[i], hin[i], d.Cr, d.Cr, T, 1, B, TC_BK, TC_BM, f16, TC_MAP_OPERAND));
    CMWG_PROPAGATE(get_slab_map(&p.g_op[i], gop[i], d.Cd, d.Cd, T, 1, B, TC_BK, TC_BM, f16, TC_MAP_OPERAND));
    CMWG_PROPAGATE(get_matrix_map(&p.pa[i], pk + PL.PA[i], d.KA, d.npadA, MEGA_BN / 2, f16));
    if (i < d.depth - 1) CMWG_PROPAGATE(get_matrix_map(&p.pb[i], pk + PL.PB[i], d.ldPB, d.nb(i), MEGA_BN / 2, f16));
    CMWG_PROPAGATE(get_slab_map(&p.g_c16[i], gop[i], d.Cd, d.Cd, T, 1, B, 32, 32, f16, TC_MAP_CHUNK16));
    if (save) CMWG_PROPAGATE(get_slab_map(&p.b_c16[i], sb[i], d.Cd, d.Cd, T, 1, B, 32, 32, f16, TC_MAP_CHUNK16));
    CMWG_PROPAGATE(get_slab_map(&p.hi_c16[i], hin[i], d.Cr, d.Cr, T, 1, B, 32, 32, f16, TC_MAP_CHUNK16));
    if (res_lo) CMWG_PROPAGATE(get_slab_map(&p.lo_c16[i], hlo[i], d.Cr, d.Cr, T, 1, B, 32, 32, f16, TC_MAP_CHUNK16));
  }
  CMWG_PROPAGATE(get_slab_map(&p.cond_op, ycl, d.auxp, d.auxp, T, 1, B, TC_BK, TC_BM, f16, TC_MAP_OPERAND));
  CMWG_PROPAGATE(get_matrix_map(&p.ps, pk + PL.PS, d.ldPS, d.Cs, MEGA_BN / 2, f16));
  CMWG_PROPAGATE(get_slab_map(&p.skip_c32, skip32, d.Cs, d.Cs, T, 1, B, 32, 32, f16, TC_MAP_CHUNK32));
  p.depth = d.depth; p.B = B; p.T = T;
  p.tiles_per_batch = ceil_div(T, 2 * TC_BM);
  p.RT = B * p.tiles_per_batch;
  if (vl.on()) {
    // only the row tiles that hold valid rows are tasks; rt -> (item, tile, tiles of the item) comes from a table on the device
    int4* tab = reinterpret_cast<int4*>(ws + varlen_tab_offset(d, B, T));
    p.RT = varlen_row_tiles(vl.host, B);
    p.rt_tab = tab;
    p.row_len = vl.dev;
    varlen_tiles_kernel<<<ceil_div(p.RT, 256), 256, 0, st>>>(vl.dev, B, T, p.RT, tab);
    CMWG_COUNT_LAUNCH();
    CMWG_LAUNCH_CHECK();
    // The taps of the last tile of an item reach up to max_dil rows past it: rows of the slab that no task of this call
    // writes and that hold whatever an earlier call left in these per-stream slabs.  Zero them in every layer-input slab.
    const int max_dil = ((d.radix - 1) / 2) << (d.depth - 1);
    dim3 zg(B, 2);
    varlen_zero_tail_kernel<<<zg, 256, 0, st>>>(vl.dev, T, max_dil, d.Cr, reinterpret_cast<uint16_t*>(hin[0]),
                                                reinterpret_cast<uint16_t*>(hin[d.depth > 1 ? 1 : 0]));
    CMWG_COUNT_LAUNCH();
    CMWG_LAUNCH_CHECK();
  }
  p.ngt = d.npadA / MEGA_BN;
  p.taps = d.R; p.kb_h = d.Crp / TC_BK; p.kb_c = d.auxp / TC_BK; p.kb_g = d.Cdp / TC_BK;
  p.Cd = d.Cd; p.f16 = f16;
  {
    const char* e = getenv("CMWG_MEGA_KTRIM");   // CMWG_MEGA_KTRIM=0: issue the padded K steps too (A/B timing)
    const int real_last = d.aux - (p.kb_c - 1) * TC_BK;
    p.kc_last = (e && e[0] == '0') ? TC_BK / 16 : std::max(1, std::min(TC_BK / 16, ceil_div(real_last, 16)));
  }
  if (fold0) {
    p.fold0 = 1;
    const int real_last0 = d.aux + d.R * d.cin - (p.kb_c - 1) * TC_BK;
    p.kc_last0 = p.kc_last == TC_BK / 16 ? p.kc_last : std::max(1, std::min(TC_BK / 16, ceil_div(real_last0, 16)));
    CMWG_PROPAGATE(get_matrix_map(&p.pa0f, pk + PL.PA0f, d.auxp, d.npadA, MEGA_BN / 2, f16));
    CMWG_PROPAGATE(get_matrix_map(&p.pb0f, pk + PL.PB0f, d.Cdp + d.kb, d.Cr, MEGA_BN / 2, f16));
  }
  p.idesc = make_idesc(f16, 2 * TC_BM, MEGA_BN, 0, 0);
  p.desc_lbo = 1u; p.desc_sbo = 1024u >> 4;
  // R(u) must come after G(u) and before G(u + RT - 1) (its right-hand neighbour one layer up): lag <= RT - 2
  p.lag = mega_fwd_lag(p.RT);
  p.dual = mega_dual();
  p.gate_mix = gate_mix();
  {
    // measured SLOWER than the TMA chunks (whole WN forward 0.540 vs 0.503 ms, saving 0.598 vs 0.560: row-per-thread 32-byte
    // accesses and a device-scope fence per lane cost more than the queueing they avoid): opt-in, kept for the comparison
    const char* e = getenv("CMWG_MEGA_RDIRECT");
    p.res_direct = (e && e[0] == '1') ? 1 : 0;
    for (int i = 0; i < d.depth; ++i) {
      p.hi_ptr[i] = reinterpret_cast<const uint16_t*>(hin[i]);
      p.hi_out_ptr[i] = reinterpret_cast<uint16_t*>(hin[i]);
      p.lo_ptr[i] = reinterpret_cast<uint16_t*>(hlo[i]);
    }
  }
  if (mega_end_fused(d)) {
    p.lst = lst;
    p.w_end = reinterpret_cast<const float*>(pk + PL.wEnd);
    p.cout = 2 * d.cin;
    // training: the `end` weight gradient reads the fp32 skip sum -- unless the backward folds the `end` conv completely
    p.store_skip = (save && !bwd_foldend_full(d, B, T)) ? 1 : 0;
  }
  p.total_tasks = (d.depth * p.RT + p.lag) * (p.ngt + 1) + p.RT;
  // timing experiments that SKIP synchronisation or epilogue work (wrong results by design) exist only in builds made
  // with -DCMWG_MEGA_EXPERIMENTS; the shipped library ignores CMWG_MEGA_DBG
#ifdef CMWG_MEGA_EXPERIMENTS
  static const int dbg_env = [] { const char* v = getenv("CMWG_MEGA_DBG"); return v ? atoi(v) : 0; }();
  p.dbg = dbg_env;
#else
  p.dbg = 0;
#endif
  // "lagged" completion signals (a unit's stores complete behind the next unit's work, its dependency counter is released one
  // unit later) were measured slower in round 1 (0.51 vs 0.476 ms at the LJ shape: consumers wait longer than the epilogue
  // warps save) and are not maintained with the scout / fused-epilogue arrangement: always immediate.
  p.lagged = 0;
  {
    // CMWG_MEGA_CLK=1: per-role cycle accumulators of the LAST launch, read back with cmwg_mega_clk_read (tools only)
    const char* v = getenv("CMWG_MEGA_CLK");
    if (v && v[0] == '1') {
      if (!g_mega_clk) CMWG_CHECK_CUDA(cudaMalloc(&g_mega_clk, (size_t)256 * 18 * 16 * sizeof(long long)));
      CMWG_CHECK_CUDA(cudaMemsetAsync(g_mega_clk, 0, (size_t)256 * 18 * 16 * sizeof(long long), st));
      p.clk = g_mega_clk;
    }
  }
  p.flags = reinterpret_cast<uint32_t*>(ws + FL.flags);
  CMWG_CHECK_CUDA(cudaMemsetAsync(p.flags, 0, (size_t)d.depth * 2 * p.RT * 4, st));
  if (vl.on()) return mega_launch<false, true>(p, st);   // inference only: no saves
  return save ? mega_launch<true>(p, st) : mega_launch<false>(p, st);
}


// single-kernel backward chain (engine_mega.cuh): dgate + dx GEMM tiles of all layers as one task list
static int wn_backward_mega(const WnDims& d, const PackedLayout& PL, const BwdLayout& BL, const uint8_t* pk, uint8_t* ws,
                            int B, int T, int f16, void* const* dh_hi, void* const* dh_lo, const void* dskip,
                            const void* dl16, void* const* dpre, const void* const* sa, const void* const* sb,
                            cudaStream_t st) {
  MegaBwdParams p;
  memset(&p, 0, sizeof(p));
  if (dl16 != nullptr) {
    p.fold_end = 1;
    p.kdl = std::max(1, ceil_div(2 * d.cin, 16));
    CMWG_PROPAGATE(get_slab_map(&p.dl_op, dl16, d.kb, d.kb, T, 1, B, TC_BK, TC_BM, f16, TC_MAP_OPERAND));
    for (int i = 0; i < d.depth; ++i)
      CMWG_PROPAGATE(get_matrix_map(&p.q1f[i], pk + PL.Q1f[i], k1f(d, i), d.Cd, MEGA_BN / 2, f16));
  }
  p.res_lo = fwd_res_lo(d) ? 1 : 0;
  for (int i = 0; i < d.depth; ++i) {
    CMWG_PROPAGATE(get_slab_map(&p.dh_op[i], dh_hi[i], d.Cr, d.Cr, T, 1, B, TC_BK, TC_BM, f16, TC_MAP_OPERAND));
    CMWG_PROPAGATE(get_slab_map(&p.dpre_op[i], dpre[i], 2 * d.Cd, 2 * d.Cd, T, 1, B, TC_BK, TC_BM, f16, TC_MAP_OPERAND));
    CMWG_PROPAGATE(get_matrix_map(&p.q1[i], pk + PL.Q1[i], d.k1(i), d.Cd, MEGA_BN / 2, f16));
    CMWG_PROPAGATE(get_matrix_map(&p.q2[i], pk + PL.Q2[i], d.ldQ2, d.Cr, MEGA_BN / 2, f16));
    CMWG_PROPAGATE(get_slab_map(&p.sa_c16[i], sa[i], d.Cd, d.Cd, T, 1, B, 32, 32, f16, TC_MAP_CHUNK16));
    CMWG_PROPAGATE(get_slab_map(&p.sb_c16[i], sb[i], d.Cd, d.Cd, T, 1, B, 32, 32, f16, TC_MAP_CHUNK16));
    // two column windows of the dpre slab (each exposes its own Cd channels)
    CMWG_PROPAGATE(get_slab_map(&p.dpt_c16[i], dpre[i], d.Cd, 2 * d.Cd, T, 1, B, 32, 32, f16, TC_MAP_CHUNK16));
    CMWG_PROPAGATE(get_slab_map(&p.dps_c16[i], (const uint16_t*)dpre[i] + d.Cd, d.Cd, 2 * d.Cd, T, 1, B, 32, 32, f16,
                                TC_MAP_CHUNK16));
    CMWG_PROPAGATE(get_slab_map(&p.dhi_c16[i], dh_hi[i], d.Cr, d.Cr, T, 1, B, 32, 32, f16, TC_MAP_CHUNK16));
    if (p.res_lo) CMWG_PROPAGATE(get_slab_map(&p.dlo_c16[i], dh_lo[i], d.Cr, d.Cr, T, 1, B, 32, 32, f16, TC_MAP_CHUNK16));
  }
  CMWG_PROPAGATE(get_slab_map(&p.dskip_op, dskip, d.Cs, d.Cs, T, 1, B, TC_BK, TC_BM, f16, TC_MAP_OPERAND));
  p.depth = d.depth; p.B = B; p.T = T;
  p.tiles_per_batch = ceil_div(T, 2 * TC_BM);
  p.RT = B * p.tiles_per_batch;
  p.taps = d.R; p.kb_r = d.Crp / TC_BK; p.kb_s = d.Csp / TC_BK; p.kb_d2 = d.Cd2p / TC_BK;
  p.f16 = f16;
  p.idesc = make_idesc(f16, 2 * TC_BM, MEGA_BN, 0, 0);
  p.desc_lbo = 1u; p.desc_sbo = 1024u >> 4;
  p.lag = mega_bwd_lag(p.RT);
  p.dual = mega_dual();
  {
    const char* e = getenv("CMWG_MEGA_RDIRECT");   // see wn_forward_mega: opt-in, measured slower
    p.direct = (e && e[0] == '1') ? 1 : 0;
    for (int i = 0; i < d.depth; ++i) {
      p.sa_ptr[i] = reinterpret_cast<const uint16_t*>(sa[i]);
      p.sb_ptr[i] = reinterpret_cast<const uint16_t*>(sb[i]);
      p.dpre_ptr[i] = reinterpret_cast<uint16_t*>(dpre[i]);
      p.dhi_ptr[i] = reinterpret_cast<uint16_t*>(dh_hi[i]);
      p.dlo_ptr[i] = reinterpret_cast<uint16_t*>(dh_lo[i]);
    }
  }
  p.total_tasks = p.RT + 2 * (d.depth * p.RT + p.lag);
  p.flags = reinterpret_cast<uint32_t*>(ws + BL.flags);
  CMWG_CHECK_CUDA(cudaMemsetAsync(p.flags, 0, (size_t)d.depth * 2 * p.RT * 4, st));
  auto kern = wn_bwd_mega_kernel;
  constexpr size_t smem = MEGA_BWD_SMEM_BYTES;
  static_assert(smem <= TC_SMEM_LIMIT, "shared memory budget exceeded");
  static bool attr_set = false;
  if (!attr_set) {
    CMWG_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set = true;
  }
  const int pairs = std::min(p.total_tasks, num_sms() / 2);
  ProfScope prof(st, CMWG_KCLASS_BWDFUSED);
  void* args[1] = {(void*)&p};
  CMWG_PROPAGATE(tc_launch_pairs_coresident((const void*)kern, smem, pairs, args, st, MEGA_THREADS));
  CMWG_COUNT_LAUNCH();
  return CMWG_OK;
}

template <typename OpT>
static int wn_forward_impl(const WnDims& d, const void* packed, const float* x, long long x_bs, const void* ycl, int B,
                           int T, void* workspace, void* saved, float* lst, cudaStream_t st, LineWin lw = LineWin(),
                           const VarLen& vl = VarLen()) {
  using E = EngineSel<OpT>;
  constexpr bool TC = E::kTc;
  const int f16 = d.prec == CMWG_PREC_FP16;
  PackedLayout PL = make_packed_layout(d);
  FwdLayout FL;
  make_fwd_layout(d, B, T, &FL);
  const uint8_t* pk = cu8(packed);
  uint8_t* ws = u8(workspace);
  uint8_t* sv = u8(saved);
  const bool save = saved != nullptr;
  CMWG_REQUIRE(!(save && lw.state), "line-window forward keeps no backward state");
  uint8_t* stt = u8(lw.state);
  const bool keep = save || stt != nullptr;  // every layer's input slab is kept (per-layer buffers)
  const size_t st_slab = line_state_slab_bytes(d, B, T);
  const int t_off = lw.nh > 0 ? lw.h0 * T : 0;             // window over the flattened (line, time) axis
  const int t_n = lw.nh > 0 ? lw.nh * T : d.H * T;

  float* h32 = reinterpret_cast<float*>(ws + FL.h32);
  float* skip32 = save ? reinterpret_cast<float*>(sv + FL.s_skip) : reinterpret_cast<float*>(ws + FL.skip32);
  // operand (16-bit hi half on the tc engine) of layer i's input
  auto hin_op = [&](int i) -> OpT* {
    if (save) return reinterpret_cast<OpT*>(sv + FL.s_hin[i]);
    if (stt) return reinterpret_cast<OpT*>(stt + (size_t)i * st_slab);
    if (TC) return reinterpret_cast<OpT*>(ws + FL.hi2[i & 1]);
    return reinterpret_cast<OpT*>(ws + FL.hop);  // ff: aliases h32
  };
  auto hlo_op = [&](int i) -> OpT* { return reinterpret_cast<OpT*>(ws + FL.lo2[i & 1]); };  // tc only
  auto g_op = [&](int i) -> OpT* {
    if (save) return reinterpret_cast<OpT*>(sv + FL.s_g[i]);
    if (TC) return reinterpret_cast<OpT*>(ws + FL.gl[i]);
    return reinterpret_cast<OpT*>(ws + FL.gop);
  };
  const int bpb = ceil_div(T, ROWS_PER_BLOCK);

  bool use_mega = false, fold0 = false;
  if constexpr (TC) {
    use_mega = mega_enabled() && !stt && lw.nh == 0 && mega_shapes_ok(d, B, T);
    fold0 = use_mega && fold0_enabled(d);
  }

  // ---- start conv (folded into layer 0's GEMM tiles when fold0: the taps of x_a go into the conditioning slab's padding)
  if (fold0) {
    const long long n = (long long)B * T * d.R * d.cin;
    const int nb_aug = (int)std::min<long long>(ceil_div_ll(n, 256), 4 * 148 * 8);
    CMWG_CHECK_CUDA(launch_pdl(cond_aug_kernel, dim3(nb_aug), dim3(256), 0, st, x, x_bs, d.cin, d.R, B, T,
                               reinterpret_cast<uint16_t*>(const_cast<void*>(ycl)), d.aux, d.auxp, f16, vl.dev));
    CMWG_COUNT_LAUNCH();
    CMWG_LAUNCH_CHECK();
  } else {
    // tc: (hi, lo) 16-bit pair; ff inference: h32 only (operand aliases it); ff training: fp32 copy per layer
    float* o32 = (!TC && !keep) ? h32 : nullptr;
    OpT* oop = (TC || keep) ? hin_op(0) : nullptr;
    OpT* olo = (TC && fwd_res_lo(d)) ? hlo_op(0) : nullptr;
    CMWG_PROPAGATE(smallk_to_slab<OpT>(x, x_bs, reinterpret_cast<const float*>(pk + PL.wStart), d.cin, 1,
                                       d.bias ? reinterpret_cast<const float*>(pk + PL.biasStart) : nullptr, d.cin,
                                       d.Cr, B, d.H * T, o32, oop, olo, f16, st, t_off, t_n, nullptr, vl.dev));
  }

  bool fused = false;
  if constexpr (TC) {
    if (use_mega) {
      void *hin[MEGA_D], *hlo[MEGA_D], *gop[MEGA_D], *sb[MEGA_D];
      for (int i = 0; i < d.depth; ++i) {
        hin[i] = hin_op(i); hlo[i] = hlo_op(i); gop[i] = g_op(i);
        sb[i] = save ? sv + FL.s_b[i] : nullptr;
      }
      CMWG_PROPAGATE(wn_forward_mega(d, PL, FL, pk, ws, ycl, B, T, save, fold0, f16, hin, hlo, gop, sb, skip32, lst, st, vl));
      fused = true;
    }
  }

  for (int i = 0; i < d.depth && !fused; ++i) {
    const int dil = 1 << i;
    const bool last = (i == d.depth - 1);
    // ---- gate GEMM
    {
      GemmDesc g;
      memset(&g, 0, sizeof(g));
      for (int s = 0; s < d.R; ++s) {
        g.seg[s].a = hin_op(i); g.seg[s].lda = d.Cr; g.seg[s].K = d.Cr;
        g.seg[s].shift = d.tap_dt(i, s); g.seg[s].shift_h = d.tap_dh(i, s); g.seg[s].koff = s * d.Crp;
      }
      g.seg[d.R].a = ycl; g.seg[d.R].lda = d.auxp; g.seg[d.R].K = d.auxp; g.seg[d.R].shift = 0;
      g.seg[d.R].koff = d.R * d.Crp;
      g.seg[d.R].bcast_h = d.H > 1;  // the conditioning has no height dimension (model/waveflow.py:131)
      g.nseg = d.R + 1;
      g.w = pk + PL.PA[i]; g.ldw = d.KA; g.N = d.npadA; g.n_rows_w = d.npadA;
      g.B = B; g.T = T; g.H = d.H; g.h0 = lw.h0; g.nh = lw.nh; g.bn = d.bn_gate; g.is_fp16 = f16; g.tag = CMWG_KCLASS_GATE;
      const float* biasA = d.bias ? reinterpret_cast<const float*>(pk + PL.biasA[i]) : nullptr;
      if constexpr (TC) {
        TcIo io;
        memset(&io, 0, sizeof(io));
        io.out[0] = op_stream(g_op(i), d.Cd);
        if (save) {
          io.out[1] = op_stream(sv + FL.s_b[i], d.Cd);   // the backward recovers tanh as g / sigmoid (GateBwdTcEpi)
          GateTcEpi<true> epi{biasA, d.Cd, f16, gate_mix()};
          CMWG_PROPAGATE(tc_gemm_launch(g, io, epi, st));
        } else {
          GateTcEpi<false> epi{biasA, d.Cd, f16, gate_mix()};
          CMWG_PROPAGATE(tc_gemm_launch(g, io, epi, st));
        }
      } else {
        GateEpi<OpT, TC> epi;
        epi.g = g_op(i);
        epi.a_save = save ? reinterpret_cast<OpT*>(sv + FL.s_a[i]) : nullptr;
        epi.b_save = save ? reinterpret_cast<OpT*>(sv + FL.s_b[i]) : nullptr;
        epi.bias = biasA;
        epi.Cd = d.Cd; epi.f16 = f16;
        CMWG_PROPAGATE((E::template gemm<true>(g, epi, st)));
      }
    }
    if constexpr (TC) {
      // ---- residual GEMM: h_{i+1} = g W_res^T + (hi_i + lo_i); the (hi, lo) pair of the layer input is
      // TMA-loaded into the epilogue and the new pair is TMA-stored
      if (!last) {
        GemmDesc g;
        memset(&g, 0, sizeof(g));
        g.seg[0].a = g_op(i); g.seg[0].lda = d.Cd; g.seg[0].K = d.Cd; g.seg[0].koff = 0;
        g.nseg = 1;
        g.w = pk + PL.PB[i]; g.ldw = d.ldPB; g.N = d.Cr; g.n_rows_w = d.nb(i);
        g.B = B; g.T = T; g.H = d.H; g.h0 = lw.h0; g.nh = lw.nh; g.bn = pick_bn(d.Cr); g.is_fp16 = f16; g.tag = CMWG_KCLASS_RESSKIP;
        g.row_len = vl.dev;
        TcIo io;
        memset(&io, 0, sizeof(io));
        const float* biasB = d.bias ? reinterpret_cast<const float*>(pk + PL.biasB[i]) : nullptr;
        io.in[0] = op_stream(hin_op(i), d.Cr);
        io.out[0] = op_stream(hin_op(i + 1), d.Cr);
        if (fwd_res_lo(d)) {
          io.in[1] = op_stream(hlo_op(i), d.Cr);
          io.out[1] = op_stream(hlo_op(i + 1), d.Cr);
          SplitTcEpi<true> epi{biasB, f16};
          CMWG_PROPAGATE(tc_gemm_launch(g, io, epi, st));
        } else {
          AddTcEpi epi{biasB, f16};   // fp16 operands: the residual stream is the operand slab alone
          CMWG_PROPAGATE(tc_gemm_launch(g, io, epi, st));
        }
      }
    } else {
      // ---- residual / skip GEMM (fp32 engine: read-modify-write epilogue)
      GemmDesc g;
      memset(&g, 0, sizeof(g));
      g.seg[0].a = g_op(i); g.seg[0].lda = d.Cd; g.seg[0].K = d.Cd; g.seg[0].shift = 0; g.seg[0].koff = 0;
      g.nseg = 1;
      g.w = pk + PL.PB[i]; g.ldw = d.ldPB; g.N = d.nb(i); g.n_rows_w = d.nb(i);
      g.B = B; g.T = T; g.H = d.H; g.h0 = lw.h0; g.nh = lw.nh; g.bn = pick_bn(d.nb(i)); g.is_fp16 = f16; g.tag = CMWG_KCLASS_RESSKIP;
      ResSkipEpi<OpT> epi;
      if (!keep) {
        epi.res_src = h32; epi.res_src_op = nullptr; epi.res_dst32 = h32; epi.res_dst_op = nullptr;
      } else {
        epi.res_src = nullptr; epi.res_src_op = hin_op(i); epi.res_dst32 = nullptr;
        epi.res_dst_op = last ? nullptr : hin_op(i + 1);
      }
      epi.skip = skip32;
      epi.bias = d.bias ? reinterpret_cast<const float*>(pk + PL.biasB[i]) : nullptr;
      epi.Cr = d.Cr; epi.Cs = d.Cs; epi.cr_eff = d.cr_eff(i); epi.first_layer = (i == 0); epi.f16 = f16;
      epi.row_len = vl.dev; epi.T = T;
      CMWG_PROPAGATE((E::template gemm<false>(g, epi, st)));
    }
  }
  if constexpr (TC) if (!fused) {
    // ---- skip GEMM: cum_skip = sum_i g_i W_skip,i^T as ONE GEMM with the layers concatenated along K
    // (accumulation across layers happens in TMEM; the fp32 result is written once)
    GemmDesc g;
    memset(&g, 0, sizeof(g));
    for (int i = 0; i < d.depth; ++i) {
      g.seg[i].a = g_op(i); g.seg[i].lda = d.Cd; g.seg[i].K = d.Cd; g.seg[i].shift = 0; g.seg[i].koff = i * d.Cdp;
    }
    g.nseg = d.depth;
    g.w = pk + PL.PS; g.ldw = d.ldPS; g.N = d.Cs; g.n_rows_w = d.Cs;
    g.B = B; g.T = T; g.H = d.H; g.h0 = lw.h0; g.nh = lw.nh; g.bn = pick_bn(d.Cs); g.is_fp16 = f16; g.tag = CMWG_KCLASS_RESSKIP;
    TcIo io;
    memset(&io, 0, sizeof(io));
    io.out[0] = f32_stream(skip32, d.Cs);
    StoreTcEpi epi{d.bias ? reinterpret_cast<const float*>(pk + PL.biasS) : nullptr, nullptr};
    CMWG_PROPAGATE(tc_gemm_launch(g, io, epi, st));
  }
  // ---- end conv (the task kernel has it in the epilogue of its skip tiles)
  if (!(fused && mega_end_fused(d))) {
    CMWG_PROPAGATE(end_fwd_launch(skip32, reinterpret_cast<const float*>(pk + PL.wEnd),
                                  d.bias ? reinterpret_cast<const float*>(pk + PL.biasEnd) : nullptr, 2 * d.cin, d.Cs, B,
                                  d.H * T, lst, st, t_off, t_n));
  }
  return CMWG_OK;
}

// ------------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------------
// fixed-order reduction of [nblocks][P] block partials into out[P]; `scratch` holds ceil(nblocks/64)*P floats
static int reduce_blocks(const float* partial, int nblocks, int P, float* scratch, float* out, cudaStream_t st,
                         const float* gscale = nullptr) {
  if (nblocks > 512) {
    int stages = ceil_div(nblocks, 64);
    reduce_blocks_stage_kernel<<<dim3(ceil_div(P, 128), stages), 128, 0, st>>>(partial, nblocks, P, scratch);
    CMWG_COUNT_LAUNCH();
    CMWG_LAUNCH_CHECK();
    partial = scratch;
    nblocks = stages;
  }
  reduce_blocks_kernel<<<ceil_div(P, 32), 256, 0, st>>>(partial, nblocks, P, out, gscale);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

// deferred weight-norm backward: every conv of the WN appends one entry, one launch at the end
struct WnBwdQueue {
  WnBwdTable tb;
  int rows = 0;
  WnBwdQueue() { tb.n = 0; }
  void add(const float* dw, const cmwg_conv_param& prm, const float* inv_norm, const cmwg_conv_grad& gr, int O, int L) {
    if (!gr.g && !gr.v) return;
    WnBwdEntry& e = tb.e[tb.n++];
    e.dw = dw; e.v = prm.v; e.g = prm.g; e.inv_norm = inv_norm; e.dg = gr.g; e.dv = gr.v; e.O = O; e.L = L;
    e.row_begin = rows;
    e.nsrc = 0;
    rows += O;
  }
  // gather `dw` from a full-K weight-gradient tile instead of a materialised matrix (see WnBwdSrc); false: no room / no entry
  bool add_source(const float* dw, const float* tile, int M, int ld, int n_valid, long long sm, long long sn, long long off) {
    for (int i = 0; i < tb.n; ++i) {
      WnBwdEntry& e = tb.e[i];
      if (e.dw != dw) continue;
      if (e.nsrc >= WN_BWD_MAX_SRC || sm != e.L || e.L > WN_BWD_MAX_L) return false;
      WnBwdSrc& sj = e.src[e.nsrc++];
      sj.tile = tile; sj.M = M; sj.ld = ld; sj.n_valid = n_valid;
      sj.row0 = (int)(off / e.L); sj.col0 = (int)(off % e.L); sj.sn = (int)sn;
      return true;
    }
    return false;
  }
  void reset() { tb.n = 0; rows = 0; }
  int flush(cudaStream_t st, const float* gscale = nullptr) {
    tb.gscale = gscale;
    if (rows == 0) return CMWG_OK;
    weight_norm_bwd_kernel<<<rows, 128, 0, st>>>(tb);
    CMWG_COUNT_LAUNCH();
    CMWG_LAUNCH_CHECK();
    return CMWG_OK;
  }
};

template <typename OpT>
static int colsum_to(const OpT* a, int ld, int C, long long rows, float* partial, float* out, int f16,
                     cudaStream_t st, const float* gscale = nullptr) {
  int nblocks = (int)ceil_div_ll(rows, ROWS_PER_BLOCK);
  colsum_partial_kernel<OpT><<<nblocks, 256, 0, st>>>(a, ld, C, rows, partial, f16);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return reduce_blocks(partial, nblocks, C, partial + (size_t)nblocks * C, out, st, gscale);
}

template <typename OpT>
static int wn_backward_impl(const WnDims& d, const cmwg_wn_params* prm, const void* packed, const float* x,
                            long long x_bs, const void* ycl, int B, int T, void* workspace, const void* saved,
                            const float* dlst, float* dx, long long dx_bs, float* dycl, const cmwg_wn_grads* gr,
                            cudaStream_t st) {
  using E = EngineSel<OpT>;
  constexpr bool TC = E::kTc;
  const int f16 = d.prec == CMWG_PREC_FP16;
  PackedLayout PL = make_packed_layout(d);
  FwdLayout FL;
  make_fwd_layout(d, B, T, &FL);
  BwdLayout BL;
  make_bwd_layout(d, B, T, &BL);
  const uint8_t* pk = cu8(packed);
  const uint8_t* sv = cu8(saved);
  uint8_t* ws = u8(workspace);
  const int TF = d.H * T;  // flattened (line, time) length of one batch item
  const long long rows = (long long)B * TF;
  const int bpb = ceil_div(TF, ROWS_PER_BLOCK);
  const int nblk = B * bpb;
  const int cout = 2 * d.cin;

  OpT* dskip_op = reinterpret_cast<OpT*>(ws + BL.dskip_op);
  float* dh32 = reinterpret_cast<float*>(ws + BL.dh32);
  OpT* dh_op = reinterpret_cast<OpT*>(ws + BL.dh_op);  // ff: aliases dh32
  OpT* dpre_op = reinterpret_cast<OpT*>(ws + BL.dpre_op);
  // tc: per-layer dpre (deferred conditioning-gradient GEMM) and (hi, lo) residual-gradient pairs
  auto dpre_l = [&](int i) -> OpT* { return TC ? reinterpret_cast<OpT*>(ws + BL.dprel[i]) : dpre_op; };
  // single-kernel chain: dgate + dx tiles of all layers in one launch; the weight-gradient GEMMs follow, so dh keeps
  // a hi slab per layer
  const bool fusedb = TC && bwd_fused_chain(d, B, T);
  auto dhi = [&](int i) -> OpT* {
    if (!TC) return dh_op;
    if (fusedb) return reinterpret_cast<OpT*>(ws + BL.dhi_l[i < d.depth ? i : d.depth - 1]);
    return reinterpret_cast<OpT*>(ws + BL.dhi2[i & 1]);
  };
  auto dlo = [&](int i) -> OpT* { return reinterpret_cast<OpT*>(ws + BL.dlo2[i & 1]); };
  // the saved state came from a forward with the start conv folded into layer 0 (same predicate as wn_forward_impl): no h_0 slab
  bool fold0 = false;
  if constexpr (TC) fold0 = mega_enabled() && mega_shapes_ok(d, B, T) && fold0_enabled(d);
  if (fold0) {
    // The taps of x_a ride in the padding columns of the conditioning slab, which all flows share: in the constant-memory mode
    // the recompute has just written them, but an activation-storing model (memory_efficient=False) ran every flow's forward
    // before the first backward, and the columns hold the LAST flow's taps by now.  They are cheap (7 us): write them again.
    const long long n = (long long)B * T * d.R * d.cin;
    const int nb_aug = (int)std::min<long long>(ceil_div_ll(n, 256), 4 * 148 * 8);
    CMWG_CHECK_CUDA(launch_pdl(cond_aug_kernel, dim3(nb_aug), dim3(256), 0, st, x, x_bs, d.cin, d.R, B, T,
                               reinterpret_cast<uint16_t*>(const_cast<void*>(ycl)), d.aux, d.auxp, f16, (const int*)nullptr));
    CMWG_COUNT_LAUNCH();
    CMWG_LAUNCH_CHECK();
  }
  int fold_pi = -1;                 // index of layer 0's conditioning weight-gradient problem (its tile holds D, fold0_dw_kernel)
  int splits_of[TC_MAX_WG];
  float* partial = reinterpret_cast<float*>(ws + BL.partial);
  float* dweff = reinterpret_cast<float*>(ws + BL.dweff);
  const float* skip32 = reinterpret_cast<const float*>(sv + FL.s_skip);
  const float* wEnd = reinterpret_cast<const float*>(pk + PL.wEnd);
  const float* wStart = reinterpret_cast<const float*>(pk + PL.wStart);
  WnBwdQueue wq;
  // 2-D WN: the conditioning is broadcast over lines, so its gradient is computed per line and summed afterwards
  float* dyl = (dycl && d.H > 1) ? reinterpret_cast<float*>(ws + BL.dycl_lines) : dycl;

  // ---- fp16 operands: the chain below runs on S * dlst, S a power of two chosen here on the device (wn_kernels.cuh)
  float* gscale = nullptr;
  if (TC && f16) {
    gscale = reinterpret_cast<float*>(ws + BL.gscale);
    CMWG_REQUIRE((reinterpret_cast<uintptr_t>(dlst) & 15) == 0, "cmwg_wn_backward: dlst must be 16-byte aligned");
    CMWG_CHECK_CUDA(cudaMemsetAsync(gscale, 0, 16, st));
    const long long n_dl = (long long)B * cout * TF;
    const int nb_gs = (int)std::max<long long>(1, std::min<long long>(ceil_div_ll(n_dl, 256 * 4 * 4), 64));
    grad_scale_kernel<<<nb_gs, 256, 0, st>>>(gscale, dlst, n_dl, wEnd, cout, d.Cs);
    CMWG_COUNT_LAUNCH();
    CMWG_LAUNCH_CHECK();
  }

  // weight-gradient GEMMs of all layers in ONE launch after the single-kernel chain
  const bool wg_batched = TC && bwd_wgrad_batched(d, B, T);
  // `end` conv folded into the backward: fe_dg -- the dgate tiles of the chain read S * dlst (one k-block) against
  // (W_end W_skip)^T instead of the 256-channel dskip slab; fe_full -- the weight gradients that dskip feeds (skip rows of every
  // W_o, the `end` weight) go through the fold as well (foldend_dw_kernel), so dskip is never formed.  CMWG_FOLD_END_W=0
  // keeps the slab for the weight gradients.
  const bool fe_dg = fusedb && foldend_enabled(d);
  const bool fe_full = TC && bwd_foldend_full(d, B, T);
  uint16_t* dl16 = nullptr;
  int p_pi[CMWG_MAX_DEPTH];
  for (int i = 0; i < CMWG_MAX_DEPTH; ++i) p_pi[i] = -1;
  if (fe_dg) {   // S * dlst as a one-k-block operand slab
    dl16 = reinterpret_cast<uint16_t*>(ws + BL.dl16);
    const int nb_dl = (int)std::min<long long>(ceil_div_ll(rows * (d.kb / 8), 256), 4 * 148 * 8);
    CMWG_CHECK_CUDA(launch_pdl(dl_slab_kernel, dim3(nb_dl), dim3(256), 0, st, dlst, cout, TF, rows, d.kb, dl16, f16,
                               (const float*)gscale));
    CMWG_COUNT_LAUNCH();
    CMWG_LAUNCH_CHECK();
  }

  // ---- end conv backward: dskip, d end.weight, d end.bias
  if (fe_full) {
    if (gr->end.v) {   // the matrix is written by foldend_dw_kernel + one reduction after the weight-gradient launch
      cmwg_conv_grad ge = gr->end;
      ge.g = nullptr;
      cmwg_conv_param pe = prm->end;
      pe.g = nullptr;
      wq.add(dweff + BL.dweff_end, pe, nullptr, ge, cout, d.Cs);
    }
  } else {
    CMWG_PROPAGATE(smallk_to_slab<OpT>(dlst, (long long)cout * TF, wEnd, 1, d.Cs, nullptr, cout, d.Cs, B, TF, nullptr,
                                       dskip_op, (OpT*)nullptr, f16, st, 0, -1, gscale));
    if (gr->end.v || gr->end.bias) {
      size_t smem2 = ((size_t)cout * ROWS_PER_BLOCK + (size_t)ROWS_PER_BLOCK * d.Cs) * sizeof(float);
      float* pw = partial;
      float* pb = partial + (size_t)nblk * cout * d.Cs;
      float* scratch = pb + (size_t)nblk * cout;
      int nblk_e = nblk;  // CTAs whose partials the reductions below fold
      float* pbe = gr->end.bias ? pb : nullptr;
      if (d.Cs == 256 && cout <= 8 && cout >= 2 && !(cout & 1)) {
        nblk_e = (int)ceil_div_ll(rows, FAST_ROWS_PER_CTA);
        switch (cout) {
          case 2: end_bwd_dw256_kernel<2><<<nblk_e, 256, 0, st>>>(dlst, skip32, TF, rows, pw, pbe); break;
          case 4: end_bwd_dw256_kernel<4><<<nblk_e, 256, 0, st>>>(dlst, skip32, TF, rows, pw, pbe); break;
          case 6: end_bwd_dw256_kernel<6><<<nblk_e, 256, 0, st>>>(dlst, skip32, TF, rows, pw, pbe); break;
          default: end_bwd_dw256_kernel<8><<<nblk_e, 256, 0, st>>>(dlst, skip32, TF, rows, pw, pbe); break;
        }
      } else {
        end_bwd_dw_kernel<<<nblk, 256, smem2, st>>>(dlst, skip32, cout, d.Cs, TF, bpb, pw, pbe);
      }
      CMWG_COUNT_LAUNCH();
      CMWG_LAUNCH_CHECK();
      cmwg_conv_grad ge = gr->end;
      ge.g = nullptr;
      cmwg_conv_param pe = prm->end;
      pe.g = nullptr;  // `end` is never weight-normed (model/waveglow.py:92)
      if (ge.v) {
        float* dEnd = dweff + BL.dweff_end;
        CMWG_PROPAGATE(reduce_blocks(pw, nblk_e, cout * d.Cs, scratch, dEnd, st));
        wq.add(dEnd, pe, nullptr, ge, cout, d.Cs);
      }
      if (gr->end.bias) {
        CMWG_PROPAGATE(reduce_blocks(pb, nblk_e, cout, scratch, gr->end.bias, st));
      }
    }
  }

  const int Lc = wgrad_chunk_len(B * d.H, T);  // FFMA engine: split-K over (batch, line, time chunk)
  const int ff_splits = B * d.H * ceil_div(T, Lc);

  if constexpr (TC) {
    if (fusedb) {
      void *hh[MEGA_D], *hl[MEGA_D], *dp[MEGA_D];
      const void *sa[MEGA_D], *sb[MEGA_D];
      for (int i = 0; i < d.depth; ++i) {
        hh[i] = dhi(i); hl[i] = dlo(i); dp[i] = dpre_l(i);
        sa[i] = sv + FL.s_g[i]; sb[i] = sv + FL.s_b[i];   // gate output and saved sigmoid (tanh = g / sigmoid)
      }
      CMWG_PROPAGATE(wn_backward_mega(d, PL, BL, pk, ws, B, T, f16, hh, hl, dskip_op, dl16, dp, sa, sb, st));
    }
  }

  // weight-gradient problems: launched per layer, or -- after the single-kernel chain -- for all layers at once
  // (63 full-K tiles fill one wave of CTA pairs without any split-K partials)
  struct RedSpec { int pi; float* out; long long sm, sn, off; int n_valid; bool no_gather; };
  struct GatherSpec { float* out; const float* tile; int M, N, n_valid; long long sm, sn, off; };
  WgradProblem pr[TC_MAX_WG];
  RedSpec rs[TC_MAX_WG];
  GatherSpec gather[TC_MAX_WG];
  int np = 0, nr = 0, ngather = 0;
  bool pending_gather = false;
  const bool deferred_gather = wg_batched && !(getenv("CMWG_WGRAD_GATHER") && getenv("CMWG_WGRAD_GATHER")[0] == '0');
  auto flush_wgrad = [&](int group) -> int {
    for (int g0 = 0; g0 < np; g0 += group) {
      const int gn = std::min(group, np - g0);
      WgradProblem* gp = pr + g0;
      int splits[TC_MAX_WG];
      if (TC) tc_wgrad_plan(gp, gn, B, d.H, T, 0, splits);
      else for (int k = 0; k < gn; ++k) splits[k] = ff_splits;
      float* pcur = partial;
      for (int k = 0; k < gn; ++k) {
        gp[k].partial = pcur;
        splits_of[g0 + k] = splits[k];
        pcur += (size_t)splits[k] * gp[k].M * gp[k].N;
      }
      CMWG_REQUIRE((size_t)((uint8_t*)pcur - (uint8_t*)partial) <= BL.partial_bytes, "wgrad partial buffer overflow");
      if (TC) {
        CMWG_PROPAGATE(tc_wgrad_launch(gp, gn, B, d.H, T, f16, st));
      } else {
        for (int k = 0; k < gn; ++k) CMWG_PROPAGATE(ff_wgrad_launch(gp[k], B, d.H, T, Lc, st));
      }
      // a problem with a single split needs no reduction, only a re-layout: the weight-norm backward gathers its tile
      // itself (WnBwdSrc); problems with several splits go through the reduce kernel below
      bool any_reduce = false;
      for (int k = 0; k < nr; ++k) {
        if (rs[k].pi < g0 || rs[k].pi >= g0 + gn) continue;
        const WgradProblem& q = pr[rs[k].pi];
        if (deferred_gather && splits[rs[k].pi - g0] == 1 && !rs[k].no_gather) {
          pending_gather = true;
          gather[ngather++] = GatherSpec{rs[k].out, q.partial, q.M, q.N, rs[k].n_valid, rs[k].sm, rs[k].sn, rs[k].off};
          rs[k].pi = -1;   // taken
        } else {
          any_reduce = true;
        }
      }
      if (!any_reduce) continue;
      WgReduceTable rt;
      rt.n = 0;
      rt.gscale = gscale;
      for (int k = 0; k < nr; ++k) {
        if (rs[k].pi < g0 || rs[k].pi >= g0 + gn) continue;
        WgReduceEntry& e = rt.e[rt.n++];
        const WgradProblem& q = pr[rs[k].pi];
        e.partial = q.partial; e.splits = splits[rs[k].pi - g0]; e.M = q.M; e.N = q.N; e.n_valid = rs[k].n_valid;
        e.out = rs[k].out; e.sm = rs[k].sm; e.sn = rs[k].sn; e.off = rs[k].off;
      }
      wgrad_reduce_kernel<<<dim3(num_sms(), rt.n), 256, 0, st>>>(rt);
      CMWG_COUNT_LAUNCH();
      CMWG_LAUNCH_CHECK();
    }
    return CMWG_OK;
  };

  for (int i = d.depth - 1; i >= 0; --i) {
    const int dil = 1 << i;
    const bool last = (i == d.depth - 1);
    const OpT* hin = reinterpret_cast<const OpT*>(sv + FL.s_hin[i]);
    const OpT* gsv = reinterpret_cast<const OpT*>(sv + FL.s_g[i]);
    OpT* dpre_i = dpre_l(i);
    const OpT* dh_next = dhi(i + 1);  // operand view of dh_{i+1} (unused for the last layer)
    // ---- dgate GEMM + gate backward epilogue -> dpre
    if (!fusedb) {
      GemmDesc g;
      memset(&g, 0, sizeof(g));
      int ns = 0;
      if (!last) {
        g.seg[ns].a = dh_next; g.seg[ns].lda = d.Cr; g.seg[ns].K = d.Cr; g.seg[ns].shift = 0; g.seg[ns].koff = 0;
        ++ns;
      }
      g.seg[ns].a = dskip_op; g.seg[ns].lda = d.Cs; g.seg[ns].K = d.Cs; g.seg[ns].shift = 0;
      g.seg[ns].koff = last ? 0 : d.Crp;
      ++ns;
      g.nseg = ns;
      g.w = pk + PL.Q1[i]; g.ldw = d.k1(i); g.N = d.Cd; g.n_rows_w = d.Cd;
      g.B = B; g.T = T; g.H = d.H; g.bn = pick_bn(d.Cd); g.is_fp16 = f16; g.tag = CMWG_KCLASS_DGATE;
      if constexpr (TC) {
        TcIo io;
        memset(&io, 0, sizeof(io));
        io.in[0] = op_stream(sv + FL.s_g[i], d.Cd);    // gate output; tanh = g / sigmoid
        io.in[1] = op_stream(sv + FL.s_b[i], d.Cd);
        // two column windows of the dpre slab: each map exposes only its own Cd channels, so a partial
        // N tile (Cd < BN) is clipped instead of spilling into the other half
        io.out[0] = TcStream{dpre_i, 2 * d.Cd, d.Cd, 0};
        io.out[1] = TcStream{dpre_i + d.Cd, 2 * d.Cd, d.Cd, 0};
        GateBwdTcEpi epi{f16};
        CMWG_PROPAGATE(tc_gemm_launch(g, io, epi, st));
      } else {
        GateBwdEpi<OpT> epi;
        epi.a_save = reinterpret_cast<const OpT*>(sv + FL.s_a[i]);
        epi.b_save = reinterpret_cast<const OpT*>(sv + FL.s_b[i]);
        epi.dpre = dpre_i; epi.Cd = d.Cd; epi.ld = 2 * d.Cd; epi.f16 = f16;
        CMWG_PROPAGATE((E::template gemm<false>(g, epi, st)));
      }
    }
    // ---- weight gradients of this layer: W_o (res rows, skip rows), W per tap, V_i
    {
      if (!wg_batched) { np = 0; nr = 0; }
      const int np_before = np;
      auto add = [&](const void* a, int lda, int M, const void* b, int ldb, int N, int shift, int shift_h, int bcast) {
        WgradProblem& q = pr[np];
        q.a = a; q.lda = lda; q.a_c0 = 0; q.M = M; q.b = b; q.ldb = ldb; q.b_c0 = 0; q.N = N; q.shift = shift;
        q.shift_h = shift_h; q.bcast_h = bcast;
        q.partial = nullptr;
        return np++;
      };
      // destinations live in this layer's dweff region, three consecutive natural-layout matrices
      float* dWo = dweff + BL.dweff_layer * (size_t)i;
      float* dW = dWo + (size_t)d.nb(i) * d.Cd;
      float* dV = dW + (size_t)2 * d.Cd * d.Cr * d.R;
      auto red = [&](int pi, float* out, long long sm, long long sn, long long off, int n_valid, bool no_gather = false) {
        rs[nr++] = RedSpec{pi, out, sm, sn, off, n_valid, no_gather};
      };
      const bool want_wo = gr->W_o[i].g || gr->W_o[i].v;
      const bool want_w = gr->W[i].g || gr->W[i].v;
      const bool want_v = gr->V.g || gr->V.v;
      if (want_wo) {
        // fe_full: the skip rows are written into dWo by foldend_dw_kernel, so the residual rows are materialised too
        // (reduce pass) instead of gathered from their tile by the weight-norm backward
        if (!last) red(add(dh_next, d.Cr, d.Cr, gsv, d.Cd, d.Cd, 0, 0, 0), dWo, d.Cd, 1, 0, d.Cd, fe_full);
        if (!fe_full)
          red(add(dskip_op, d.Cs, d.Cs, gsv, d.Cd, d.Cd, 0, 0, 0), dWo, d.Cd, 1, (long long)d.cr_eff(i) * d.Cd, d.Cd);
      }
      if (fe_full) {   // (every layer, wanted or not: dW_end sums over all of them) P_i = g_i^T (S dlst): tile [Cd][kb], folded
        p_pi[i] = add(gsv, d.Cd, d.Cd, dl16, d.kb, d.kb, 0, 0, 0);   // (and unscaled) into pred[i][Cd][cout] by the reduce pass
        red(p_pi[i], reinterpret_cast<float*>(ws + BL.pred) + (size_t)i * d.Cd * cout, cout, 1, 0, cout, true);
      }
      const bool folded = fold0 && i == 0;   // no h_0 slab: dW_0 comes out of the conditioning problem's tile (fold0_dw_kernel)
      if (want_w && !folded)
        for (int s = 0; s < d.R; ++s)
          red(add(dpre_i, 2 * d.Cd, 2 * d.Cd, hin, d.Cr, d.Cr, d.tap_dt(i, s), d.tap_dh(i, s), 0), dW,
              (long long)d.Cr * d.R, d.R, s, d.Cr);
      if (want_v || (folded && want_w)) {
        const int pi = add(dpre_i, 2 * d.Cd, 2 * d.Cd, ycl, d.auxp, d.auxp, 0, 0, d.H > 1);
        if (want_v) red(pi, dV, d.aux, 1, 0, d.aux);
        if (folded && want_w) fold_pi = pi;
      }
      if (!wg_batched) CMWG_PROPAGATE(flush_wgrad(TC_WG_GROUP));
      if (np > np_before) {
        if (want_wo)
          wq.add(dWo, prm->W_o[i], reinterpret_cast<const float*>(pk + PL.nWo[i]), gr->W_o[i], d.nb(i), d.Cd);
        if (want_w)
          wq.add(dW, prm->W[i], reinterpret_cast<const float*>(pk + PL.nW[i]), gr->W[i], 2 * d.Cd, d.Cr * d.R);
        if (want_v) {
          size_t ro = (size_t)i * 2 * d.Cd;
          cmwg_conv_param pv{prm->V.g ? prm->V.g + ro : nullptr, prm->V.v + ro * d.aux, nullptr};
          cmwg_conv_grad gv{gr->V.g ? gr->V.g + ro : nullptr, gr->V.v ? gr->V.v + ro * d.aux : nullptr, nullptr};
          wq.add(dV, pv, reinterpret_cast<const float*>(pk + PL.nV) + ro, gv, 2 * d.Cd, d.aux);
        }
      }
    }
    // ---- bias gradients (bias=True only)
    if (d.bias) {
      // W_i.bias and V.bias[i] both receive the column sums of dpre
      if (gr->W[i].bias)
        CMWG_PROPAGATE(colsum_to<OpT>(dpre_i, 2 * d.Cd, 2 * d.Cd, rows, partial, gr->W[i].bias, f16, st, gscale));
      if (gr->V.bias)
        CMWG_PROPAGATE(colsum_to<OpT>(dpre_i, 2 * d.Cd, 2 * d.Cd, rows, partial, gr->V.bias + (size_t)i * 2 * d.Cd, f16, st,
                                      gscale));
      if (gr->W_o[i].bias) {
        if (!last) CMWG_PROPAGATE(colsum_to<OpT>(dh_next, d.Cr, d.Cr, rows, partial, gr->W_o[i].bias, f16, st, gscale));
        CMWG_PROPAGATE(colsum_to<OpT>(dskip_op, d.Cs, d.Cs, rows, partial, gr->W_o[i].bias + d.cr_eff(i), f16, st, gscale));
      }
    }
    // ---- conditioning gradient (fp32 engine: accumulate per layer; tc: one deferred GEMM after the loop)
    if (dycl && !TC) {
      GemmDesc g;
      memset(&g, 0, sizeof(g));
      g.seg[0].a = dpre_i; g.seg[0].lda = 2 * d.Cd; g.seg[0].K = 2 * d.Cd; g.seg[0].shift = 0; g.seg[0].koff = i * d.Cd2p;
      g.nseg = 1;
      g.w = pk + PL.QV[0]; g.ldw = d.ldQV; g.N = d.auxp; g.n_rows_w = d.auxp;
      g.B = B; g.T = T; g.H = d.H; g.bn = pick_bn(d.auxp); g.is_fp16 = f16; g.tag = CMWG_KCLASS_DCOND;
      AccumEpi epi{dyl, d.auxp, d.auxp, last ? 1 : 0};
      CMWG_PROPAGATE((E::template gemm<false>(g, epi, st)));
    }
    // ---- dx GEMM: dh_i = dh_{i+1} + conv^T(dpre)
    if (!fusedb) {
      GemmDesc g;
      memset(&g, 0, sizeof(g));
      for (int s = 0; s < d.R; ++s) {
        g.seg[s].a = dpre_i; g.seg[s].lda = 2 * d.Cd; g.seg[s].K = 2 * d.Cd;
        g.seg[s].shift = -d.tap_dt(i, s); g.seg[s].shift_h = -d.tap_dh(i, s); g.seg[s].koff = s * d.Cd2p;
      }
      g.nseg = d.R;
      g.w = pk + PL.Q2[i]; g.ldw = d.ldQ2; g.N = d.Cr; g.n_rows_w = d.Cr;
      g.B = B; g.T = T; g.H = d.H; g.bn = pick_bn(d.Cr); g.is_fp16 = f16; g.tag = CMWG_KCLASS_DX;
      if constexpr (TC) {
        TcIo io;
        memset(&io, 0, sizeof(io));
        io.out[0] = op_stream(dhi(i), d.Cr);
        if (!fwd_res_lo(d)) {   // fp16 operands: the residual gradient is the operand slab alone
          if (!last) {
            io.in[0] = op_stream(dhi(i + 1), d.Cr);
            AddTcEpiT<2> epi{nullptr, f16};
            CMWG_PROPAGATE(tc_gemm_launch(g, io, epi, st));
          } else {
            RoundTcEpi epi{f16};
            CMWG_PROPAGATE(tc_gemm_launch(g, io, epi, st));
          }
        } else {
          io.out[1] = op_stream(dlo(i), d.Cr);
          if (!last) {  // the upstream residual gradient (hi, lo) is added in the epilogue
            io.in[0] = op_stream(dhi(i + 1), d.Cr);
            io.in[1] = op_stream(dlo(i + 1), d.Cr);
            SplitTcEpi<true, 2> epi{nullptr, f16};  // K = R*2Cd is long: trade epilogue width for operand stages
            CMWG_PROPAGATE(tc_gemm_launch(g, io, epi, st));
          } else {
            SplitTcEpi<false> epi{nullptr, f16};
            CMWG_PROPAGATE(tc_gemm_launch(g, io, epi, st));
          }
        }
      } else {
        DxEpi<OpT> epi;
        epi.src = last ? nullptr : dh32; epi.dst32 = dh32; epi.dst_op = nullptr;
        epi.Cr = d.Cr; epi.f16 = f16;
        CMWG_PROPAGATE((E::template gemm<false>(g, epi, st)));
      }
    }
  }

  if (wg_batched) CMWG_PROPAGATE(flush_wgrad(TC_MAX_WG));
  if (fe_full) {
    FoldEndDwParams fp;
    memset(&fp, 0, sizeof(fp));
    bool all = true;
    for (int i = 0; i < d.depth; ++i) {
      if (p_pi[i] < 0) { all = false; break; }
      fp.wWo[i] = reinterpret_cast<const float*>(pk + PL.wWo[i]);
      fp.dWo_skip[i] = dweff + BL.dweff_layer * (size_t)i + (size_t)d.cr_eff(i) * d.Cd;
    }
    if (all) {   // (all or none: every W_o and the `end` weight of a WN are trained together)
      float* dEnd_part = reinterpret_cast<float*>(ws + BL.partial_start);   // [depth][cout][Cs], folded below
      fp.wEnd = wEnd;
      fp.pred = reinterpret_cast<const float*>(ws + BL.pred);
      fp.dEnd_part = gr->end.v ? dEnd_part : nullptr;
      fp.depth = d.depth; fp.Cd = d.Cd; fp.Cs = d.Cs; fp.Cr = d.Cr; fp.cout = cout;
      foldend_dw_kernel<<<dim3(d.Cs / FOLDEND_DW_ROWS, d.depth), 256, 0, st>>>(fp);
      CMWG_COUNT_LAUNCH();
      CMWG_LAUNCH_CHECK();
      if (gr->end.v)
        CMWG_PROPAGATE(reduce_blocks(dEnd_part, d.depth, cout * d.Cs, dEnd_part + (size_t)d.depth * cout * d.Cs,
                                     dweff + BL.dweff_end, st));
    }
  }
  if (fold_pi >= 0) {
    // layer 0's group was the last one flushed: its tiles are still in the `partial` workspace
    const WgradProblem& q = pr[fold_pi];
    fold0_dw_kernel<<<2 * d.Cd, 256, 0, st>>>(q.partial, splits_of[fold_pi], q.M, q.N, d.aux, d.cin, d.R, d.Cr, wStart, gscale,
                                              dweff + (size_t)d.nb(0) * d.Cd);
    CMWG_COUNT_LAUNCH();
    CMWG_LAUNCH_CHECK();
  }
  if (pending_gather) {
    // every destination matrix has its weight-norm entry by now: attach the tiles; leftovers go through one reduce launch
    WgReduceTable rt;
    rt.n = 0;
    rt.gscale = gscale;
    for (int k = 0; k < ngather; ++k) {
      const GatherSpec& gs = gather[k];
      if (wq.add_source(gs.out, gs.tile, gs.M, gs.N, gs.n_valid, gs.sm, gs.sn, gs.off)) continue;
      WgReduceEntry& e = rt.e[rt.n++];
      e.partial = gs.tile; e.splits = 1; e.M = gs.M; e.N = gs.N; e.n_valid = gs.n_valid;
      e.out = gs.out; e.sm = gs.sm; e.sn = gs.sn; e.off = gs.off;
    }
    if (rt.n > 0) {
      wgrad_reduce_kernel<<<dim3(num_sms(), rt.n), 256, 0, st>>>(rt);
      CMWG_COUNT_LAUNCH();
      CMWG_LAUNCH_CHECK();
    }
    // the tiles live in the `partial` workspace until the weight-norm backward at the end gathers them: the start conv
    // backward below keeps its block partials in a region of its own (BwdLayout::partial_start)
  }

  if constexpr (TC) {
    // ---- conditioning gradient: dy = sum_i dpre_i V_i as ONE GEMM, layers concatenated along K
    if (dycl) {
      GemmDesc g;
      memset(&g, 0, sizeof(g));
      for (int i = 0; i < d.depth; ++i) {
        g.seg[i].a = dpre_l(i); g.seg[i].lda = 2 * d.Cd; g.seg[i].K = 2 * d.Cd; g.seg[i].shift = 0;
        g.seg[i].koff = i * d.Cd2p;
      }
      g.nseg = d.depth;
      g.w = pk + PL.QV[0]; g.ldw = d.ldQV; g.N = d.auxp; g.n_rows_w = d.auxp;
      g.B = B; g.T = T; g.H = d.H; g.bn = pick_bn(d.auxp); g.is_fp16 = f16; g.tag = CMWG_KCLASS_DCOND;
      TcIo io;
      memset(&io, 0, sizeof(io));
      io.out[0] = f32_stream(dyl, d.auxp);
      StoreTcEpi epi{nullptr, gscale};
      CMWG_PROPAGATE(tc_gemm_launch(g, io, epi, st));
    }
  }
  if (dycl && d.H > 1) {
    long long n4 = (long long)T * d.auxp / 4;  // auxp is a multiple of 16
    dim3 grid((unsigned)std::min<long long>(ceil_div_ll(n4, 256), 4096), B);
    sum_lines_kernel<<<grid, 256, 0, st>>>(dyl, dycl, d.H, n4);
    CMWG_COUNT_LAUNCH();
    CMWG_LAUNCH_CHECK();
  }

  // ---- start conv backward
  {
    size_t smem = ((size_t)ROWS_PER_BLOCK * (d.Cr + 1) + (size_t)d.cin * ROWS_PER_BLOCK) * sizeof(float);
    float* pw = reinterpret_cast<float*>(ws + BL.partial_start);
    float* pb = pw + (size_t)nblk * d.Cr * d.cin;
    float* scratch = pb + (size_t)nblk * d.Cr;
    const float* a32 = TC ? nullptr : dh32;
    const uint16_t* ahi = TC ? reinterpret_cast<const uint16_t*>(dhi(0)) : nullptr;
    const uint16_t* alo = (TC && fwd_res_lo(d)) ? reinterpret_cast<const uint16_t*>(dlo(0)) : nullptr;
    float* pbs = (d.bias && gr->start.bias) ? pb : nullptr;
    int nblk_s = nblk;
    if (d.Cr == 256 && d.cin >= 1 && d.cin <= 8) {
      nblk_s = (int)ceil_div_ll(rows, FAST_ROWS_PER_CTA);
#define CMWG_START_CASE(N) \
  case N: start_bwd256_kernel<N><<<nblk_s, 256, 0, st>>>(a32, ahi, alo, x, x_bs, wStart, TF, rows, dx, dx_bs, pw, pbs, f16, gscale); break;
      switch (d.cin) {
        CMWG_START_CASE(1) CMWG_START_CASE(2) CMWG_START_CASE(3) CMWG_START_CASE(4)
        CMWG_START_CASE(5) CMWG_START_CASE(6) CMWG_START_CASE(7) CMWG_START_CASE(8)
      }
#undef CMWG_START_CASE
    } else {
      start_bwd_kernel<<<nblk, 256, smem, st>>>(a32, ahi, alo, x, x_bs, wStart, d.cin, d.Cr, TF, bpb, dx, dx_bs, pw, pbs, f16,
                                                gscale);
    }
    CMWG_COUNT_LAUNCH();
    CMWG_LAUNCH_CHECK();
    if (gr->start.g || gr->start.v) {
      float* dStart = dweff + BL.dweff_start;
      CMWG_PROPAGATE(reduce_blocks(pw, nblk_s, d.Cr * d.cin, scratch, dStart, st));
      wq.add(dStart, prm->start, reinterpret_cast<const float*>(pk + PL.nStart), gr->start, d.Cr, d.cin);
    }
    if (d.bias && gr->start.bias) {
      CMWG_PROPAGATE(reduce_blocks(pb, nblk_s, d.Cr, scratch, gr->start.bias, st));
    }
  }
  return wq.flush(st, gscale);
}

}  // namespace cmwg

using namespace cmwg;

extern "C" {

int cmwg_wn_tc_supported(const cmwg_wn_config* cfg) { return cfg && wn_tc_shapes_ok(*cfg) ? 1 : 0; }

int cmwg_wn_aux_padded(const cmwg_wn_config* cfg) {
  WnDims d;
  if (make_dims(cfg, &d) != CMWG_OK) return -1;
  return d.auxp;
}

size_t cmwg_wn_packed_bytes(const cmwg_wn_config* cfg) {
  WnDims d;
  if (make_dims(cfg, &d) != CMWG_OK) return 0;
  return make_packed_layout(d).total;
}

// host-side listing of the task kernels' lists (the same decode functions the kernels run): entry i -> out[4*i .. 4*i+3] =
// (type, layer, row tile, N tile); forward types 0 gate / 1 residual / 2 skip / 3 none, backward types 0 dgate / 1 dx / 3 none
int cmwg_mega_task_list(int backward, int depth, int B, int T, int* out, int cap, int* total, int* lag) {
  CMWG_REQUIRE(depth >= 1 && depth <= cmwg::MEGA_D && B >= 1 && T >= 1 && out && total && lag, "cmwg_mega_task_list: bad arguments");
  const int tpb = cmwg::ceil_div(T, 2 * cmwg::TC_BM), RT = B * tpb;
  if (backward) {
    cmwg::MegaBwdParams p;
    memset(&p, 0, sizeof(p));
    p.depth = depth; p.B = B; p.T = T; p.tiles_per_batch = tpb; p.RT = RT;
    p.lag = cmwg::mega_bwd_lag(RT);
    p.total_tasks = RT + 2 * (depth * RT + p.lag);
    *total = p.total_tasks; *lag = p.lag;
    for (int i = 0; i < p.total_tasks && i < cap; ++i) {
      const cmwg::MegaTask t = cmwg::mega_bwd_decode(p, i);
      out[4 * i] = t.type; out[4 * i + 1] = t.layer; out[4 * i + 2] = t.rt; out[4 * i + 3] = t.nt;
    }
  } else {
    cmwg::MegaParams p;
    memset(&p, 0, sizeof(p));
    p.depth = depth; p.B = B; p.T = T; p.tiles_per_batch = tpb; p.RT = RT; p.ngt = 2;
    p.lag = cmwg::mega_fwd_lag(RT);
    p.total_tasks = (depth * RT + p.lag) * (p.ngt + 1) + RT;
    *total = p.total_tasks; *lag = p.lag;
    for (int i = 0; i < p.total_tasks && i < cap; ++i) {
      const cmwg::MegaTask t = cmwg::mega_decode(p, i);
      out[4 * i] = t.type; out[4 * i + 1] = t.layer; out[4 * i + 2] = t.rt; out[4 * i + 3] = t.nt;
    }
  }
  return CMWG_OK;
}

int cmwg_mega_clk_read(long long* host, int n) {
  if (!cmwg::g_mega_clk) return CMWG_ERR_ARG;
  cudaError_t e = cudaMemcpy(host, cmwg::g_mega_clk, (size_t)n * sizeof(long long), cudaMemcpyDeviceToHost);
  return e == cudaSuccess ? CMWG_OK : CMWG_ERR_CUDA;
}

size_t cmwg_wn_workspace_bytes(const cmwg_wn_config* cfg, int B, int T) {
  WnDims d;
  if (make_dims(cfg, &d) != CMWG_OK) return 0;
  FwdLayout FL;
  make_fwd_layout(d, B, T, &FL);
  BwdLayout BL;
  make_bwd_layout(d, B, T, &BL);
  return (FL.ws_total > BL.total ? FL.ws_total : BL.total) + 1024;
}

size_t cmwg_wn_saved_bytes(const cmwg_wn_config* cfg, int B, int T) {
  WnDims d;
  if (make_dims(cfg, &d) != CMWG_OK) return 0;
  FwdLayout FL;
  make_fwd_layout(d, B, T, &FL);
  return FL.saved_total + 1024;
}

int cmwg_wn_pack(const cmwg_wn_config* cfg, const cmwg_wn_params* params, void* packed, void* stream) {
  WnDims d;
  CMWG_PROPAGATE(make_dims(cfg, &d));
  CMWG_REQUIRE(params && packed, "cmwg_wn_pack: null argument");
  return wn_pack_impl(d, params, packed, (cudaStream_t)stream);
}

int cmwg_cond_pack(const cmwg_wn_config* cfg, const float* y, long long y_bstride, long long y_cstride,
                   long long y_tstride, int B, int T, void* ycl, void* stream) {
  WnDims d;
  CMWG_PROPAGATE(make_dims(cfg, &d));
  if (B == 0 || T == 0) return CMWG_OK;
  dim3 grid(ceil_div(T, 32), ceil_div(d.auxp, 32), B);
  if (d.tc)
    cond_pack_kernel<uint16_t><<<grid, 256, 0, (cudaStream_t)stream>>>(y, y_bstride, y_cstride, y_tstride, d.aux, d.auxp,
                                                                       T, (uint16_t*)ycl, d.prec == CMWG_PREC_FP16);
  else
    cond_pack_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(y, y_bstride, y_cstride, y_tstride, d.aux, d.auxp, T,
                                                                    (float*)ycl, 0);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

int cmwg_cond_unpack_grad(const cmwg_wn_config* cfg, const float* dycl, int B, int T, float* dy, void* stream) {
  WnDims d;
  CMWG_PROPAGATE(make_dims(cfg, &d));
  if (B == 0 || T == 0) return CMWG_OK;
  dim3 grid(ceil_div(T, 32), ceil_div(d.auxp, 32), B);
  cond_unpack_grad_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(dycl, d.aux, d.auxp, T, dy);
  CMWG_COUNT_LAUNCH();
  CMWG_LAUNCH_CHECK();
  return CMWG_OK;
}

int cmwg_wn_forward(const cmwg_wn_config* cfg, const void* packed, const float* x, long long x_bstride,
                    const void* ycl, int B, int T, void* workspace, void* saved, float* lst, void* stream) {
  WnDims d;
  CMWG_PROPAGATE(make_dims(cfg, &d));
  CMWG_REQUIRE(packed && x && ycl && workspace && lst, "cmwg_wn_forward: null argument");
  if (B == 0 || T == 0) return CMWG_OK;
  if (d.tc) return wn_forward_impl<uint16_t>(d, packed, x, x_bstride, ycl, B, T, workspace, saved, lst, (cudaStream_t)stream);
  return wn_forward_impl<float>(d, packed, x, x_bstride, ycl, B, T, workspace, saved, lst, (cudaStream_t)stream);
}

size_t cmwg_wn_varlen_workspace_bytes(const cmwg_wn_config* cfg, int B, int T) {
  WnDims d;
  if (make_dims(cfg, &d) != CMWG_OK || B < 1 || T < 1) return 0;
  return varlen_tab_offset(d, B, T) + align_up((size_t)B * ceil_div(T, 2 * TC_BM) * sizeof(int4), 1024) + 1024;
}

int cmwg_wn_forward_varlen(const cmwg_wn_config* cfg, const void* packed, const float* x, long long x_bstride,
                           const void* ycl, int B, int T, const int* lengths_host, const int* lengths_dev, void* workspace,
                           float* lst, void* stream) {
  WnDims d;
  CMWG_PROPAGATE(make_dims(cfg, &d));
  CMWG_REQUIRE(packed && x && ycl && workspace && lst && lengths_host && lengths_dev, "cmwg_wn_forward_varlen: null argument");
  if (B == 0 || T == 0) return CMWG_OK;
  for (int b = 0; b < B; ++b)
    CMWG_REQUIRE(lengths_host[b] >= 1 && lengths_host[b] <= T, "cmwg_wn_forward_varlen: length %d of item %d outside [1, %d]",
                 lengths_host[b], b, T);
  if (d.H != 1) {
    set_error("cmwg_wn_forward_varlen: per-item lengths are implemented for the 1-D WN only");
    return CMWG_ERR_UNSUPPORTED;
  }
  if (d.tc && fwd_res_lo(d)) {
    const char* e = getenv("CMWG_MEGA_RDIRECT");
    if (e && e[0] == '1' && mega_enabled() && mega_shapes_ok(d, B, T)) {
      set_error("cmwg_wn_forward_varlen: CMWG_MEGA_RDIRECT=1 residual tiles do not mask rows past an item's end");
      return CMWG_ERR_UNSUPPORTED;
    }
  }
  VarLen vl;
  vl.host = lengths_host; vl.dev = lengths_dev;
  cudaStream_t st = (cudaStream_t)stream;
  if (d.tc) return wn_forward_impl<uint16_t>(d, packed, x, x_bstride, ycl, B, T, workspace, nullptr, lst, st, LineWin(), vl);
  return wn_forward_impl<float>(d, packed, x, x_bstride, ycl, B, T, workspace, nullptr, lst, st, LineWin(), vl);
}

int cmwg_mega_task_list_varlen(int depth, int B, int T, const int* lengths, int* out, int cap, int* total, int* lag, int* tiles,
                               int tiles_cap, int* row_tiles) {
  CMWG_REQUIRE(depth >= 1 && depth <= cmwg::MEGA_D && B >= 1 && T >= 1 && lengths && out && total && lag && tiles && row_tiles,
               "cmwg_mega_task_list_varlen: bad arguments");
  for (int b = 0; b < B; ++b)
    CMWG_REQUIRE(lengths[b] >= 1 && lengths[b] <= T, "cmwg_mega_task_list_varlen: length %d of item %d outside [1, %d]",
                 lengths[b], b, T);
  cmwg::MegaParams p;
  memset(&p, 0, sizeof(p));
  p.depth = depth; p.B = B; p.T = T; p.tiles_per_batch = cmwg::ceil_div(T, 2 * cmwg::TC_BM);
  p.RT = varlen_row_tiles(lengths, B);
  p.ngt = 2;
  p.lag = cmwg::mega_fwd_lag(p.RT);
  p.total_tasks = (depth * p.RT + p.lag) * (p.ngt + 1) + p.RT;
  *total = p.total_tasks; *lag = p.lag; *row_tiles = p.RT;
  for (int i = 0; i < p.total_tasks && i < cap; ++i) {
    const cmwg::MegaTask t = cmwg::mega_decode(p, i);
    out[4 * i] = t.type; out[4 * i + 1] = t.layer; out[4 * i + 2] = t.rt; out[4 * i + 3] = t.nt;
  }
  for (int b = 0, rt = 0; b < B; ++b) {   // the table varlen_tiles_kernel builds on the device
    const int n = cmwg::ceil_div(lengths[b], 2 * cmwg::TC_BM);
    for (int k = 0; k < n; ++k, ++rt)
      if (rt < tiles_cap) { tiles[3 * rt] = b; tiles[3 * rt + 1] = k; tiles[3 * rt + 2] = n; }
  }
  return CMWG_OK;
}

size_t cmwg_wn_line_state_bytes(const cmwg_wn_config* cfg, int B, int T) {
  WnDims d;
  if (make_dims(cfg, &d) != CMWG_OK) return 0;
  return (size_t)d.depth * line_state_slab_bytes(d, B, T) + 1024;
}

int cmwg_wn_forward_lines(const cmwg_wn_config* cfg, const void* packed, const float* x, long long x_bstride,
                          const void* ycl, int B, int T, int line_begin, int line_count, void* workspace, void* state,
                          float* lst, void* stream) {
  WnDims d;
  CMWG_PROPAGATE(make_dims(cfg, &d));
  CMWG_REQUIRE(packed && x && ycl && workspace && state && lst, "cmwg_wn_forward_lines: null argument");
  CMWG_REQUIRE(line_begin >= 0 && line_count >= 0 && line_begin + line_count <= d.H,
               "cmwg_wn_forward_lines: lines [%d, %d) outside [0, %d)", line_begin, line_begin + line_count, d.H);
  if (B == 0 || T == 0 || line_count == 0) return CMWG_OK;
  LineWin lw;
  lw.state = state; lw.h0 = line_begin; lw.nh = line_count;
  if (d.tc)
    return wn_forward_impl<uint16_t>(d, packed, x, x_bstride, ycl, B, T, workspace, nullptr, lst, (cudaStream_t)stream, lw);
  return wn_forward_impl<float>(d, packed, x, x_bstride, ycl, B, T, workspace, nullptr, lst, (cudaStream_t)stream, lw);
}

int cmwg_waveflow_inverse_flow(const cmwg_wn_config* cfg, const void* packed, const float* z, int in_flip,
                               const void* ycl, int B, int W, void* workspace, void* state, float* lst, float* x,
                               void* stream) {
  WnDims d;
  CMWG_PROPAGATE(make_dims(cfg, &d));
  CMWG_REQUIRE(d.H > 1 && d.cin == 1, "cmwg_waveflow_inverse_flow: needs the 2-D WN (height > 1, one input channel)");
  CMWG_REQUIRE(packed && z && ycl && workspace && state && lst && x, "cmwg_waveflow_inverse_flow: null argument");
  if (B == 0 || W == 0) return CMWG_OK;
  const int H = d.H + 1;  // image lines; the WN sees lines 0..H-2
  cudaStream_t st = (cudaStream_t)stream;
  // line 0 passes through (xnew = z[:, :, :1], model/waveflow.py:240)
  CMWG_PROPAGATE(cmwg_waveflow_affine(z, in_flip, nullptr, x, 0, B, H, W, 0, 1, 1, stream));
  LineWin lw;
  lw.state = state; lw.nh = 1;
  for (int i = 1; i < H; ++i) {  // row i from rows < i (:245-258)
    lw.h0 = i - 1;
    if (d.tc)
      CMWG_PROPAGATE(wn_forward_impl<uint16_t>(d, packed, x, (long long)H * W, ycl, B, W, workspace, nullptr, lst, st, lw));
    else
      CMWG_PROPAGATE(wn_forward_impl<float>(d, packed, x, (long long)H * W, ycl, B, W, workspace, nullptr, lst, st, lw));
    CMWG_PROPAGATE(cmwg_waveflow_affine(z, in_flip, lst, x, 0, B, H, W, i, 1, 1, stream));
  }
  return CMWG_OK;
}

int cmwg_wn_backward(const cmwg_wn_config* cfg, const cmwg_wn_params* params, const void* packed, const float* x,
                     long long x_bstride, const void* ycl, int B, int T, void* workspace, const void* saved,
                     const float* dlst, float* dx, long long dx_bstride, float* dycl, const cmwg_wn_grads* grads,
                     void* stream) {
  WnDims d;
  CMWG_PROPAGATE(make_dims(cfg, &d));
  CMWG_REQUIRE(params && packed && x && ycl && workspace && saved && dlst && dx && grads,
               "cmwg_wn_backward: null argument");
  if (B == 0 || T == 0) return CMWG_OK;
  if (d.tc)
    return wn_backward_impl<uint16_t>(d, params, packed, x, x_bstride, ycl, B, T, workspace, saved, dlst, dx, dx_bstride,
                                      dycl, grads, (cudaStream_t)stream);
  return wn_backward_impl<float>(d, params, packed, x, x_bstride, ycl, B, T, workspace, saved, dlst, dx, dx_bstride, dycl,
                                 grads, (cudaStream_t)stream);
}

}  // extern "C"
