// tcgen05 / TMEM / TMA GEMM engine for sm_100a (hand-written PTX; no CUTLASS).
//
// Persistent, warp-specialised CTAs, launched as CTA PAIRS (clusters of 2, one pair per TPC):
//   warp 0 (one lane)  TMA producer: cp.async.bulk.tensor loads into a STAGES-deep shared-memory ring
//                      (128B swizzle).  Each CTA of a pair loads ITS 128 rows of A and ITS HALF of the
//                      B (weight) tile; both signal the LEADER CTA's full barrier.
//   warp 1 (one lane)  MMA issuer (leader CTA only): tcgen05.mma.cta_group::2.kind::f16, M = 256
//                      (128 rows per CTA), N = BN, K = 16 per instruction; fp32 accumulators in the
//                      TMEM of both SMs, double buffered (2 x BN columns).  Operand traffic per flop
//                      (L2 -> shared memory and shared memory -> tensor core) is 2/3 of the 1-CTA form,
//                      which is what bounds a 128 x 256 x 64 1-CTA tile.
//   warps 2..17        epilogue (four warps per TMEM lane quadrant, a quarter of the columns each; 4 warps
//                      per scheduler hide the MUFU / conversion latencies of the fused functors):
//                      tcgen05.ld 32 lanes x 16 columns (one accumulator ROW per thread) -> fused
//                      epilogue functor -> swizzled shared-memory staging -> TMA store of 32 x 32 chunks.
//                      Epilogue INPUTS (saved gate values, residual hi/lo pairs) arrive the same way in
//                      reverse: TMA load into per-warp staging, issued one chunk ahead.  The TMA unit
//                      clips rows >= T and columns >= C on stores and zero-fills them on loads, so the
//                      epilogue has no bounds checks and no global address arithmetic.
// Pipelines: smem full/empty mbarriers (TMA <-> MMA; empty is signalled in both CTAs by a multicast
// tcgen05.commit) and TMEM full/empty mbarriers (MMA <-> epilogue; the peer's epilogue warps arrive
// remotely on the leader's tmem_empty barrier).
//
// Two operand arrangements:
//   KMAJOR  (forward / dgrad GEMMs)  A = slab rows x channels (K = channels contiguous),
//           a dilated tap is a row shift of the TMA coordinate, out-of-range rows are zero filled by
//           the TMA unit (the conv's 'same' padding);  B = packed weights [N][K].
//   MNMAJOR (weight-gradient GEMMs)  A = slab[t][m], B = slab[t + shift][n], K = time: the very
//           same slabs read through MN-major UMMA descriptors, split-K over time chunks.
#pragma once
#include <cuda.h>

#include "common.cuh"
#include "engine_ff.cuh"  // GemmDesc / WgradProblem

namespace cmwg {

constexpr int TC_BM = 128;                // rows per CTA (the pair covers 256)
constexpr int TC_BK = 64;                 // 64 x 16-bit = 128 B = one swizzle row
constexpr int TC_A_BYTES = TC_BM * 128;   // 16 KB
constexpr int TC_EPI_WARPS = 16;          // 4 per TMEM lane quadrant, each owning a quarter of the tile's columns
constexpr int TC_THREADS = 64 + 32 * TC_EPI_WARPS;
constexpr int TC_MAX_WG = 48;             // weight-gradient problems per launch (all layers of one WN at once)
constexpr int TC_WG_GROUP = 8;            // problems per launch of the layer-at-a-time pipeline
constexpr int TC_MAX_OUT = 3;             // output streams of one epilogue
constexpr int TC_MAX_IN = 2;              // input streams of one epilogue
constexpr int TC_SMEM_LIMIT = 232448;     // 227 KB opt-in shared memory per CTA

// one epilogue stream: a channel-last slab [B*T][ld] of 16-bit operands or fp32
struct TcStream {
  const void* ptr;
  int ld;      // row pitch in elements
  int cols;    // valid channels (TMA clips stores / zero-fills loads beyond them)
  int is_f32;
};
struct TcIo {
  TcStream out[TC_MAX_OUT];
  TcStream in[TC_MAX_IN];
};

struct alignas(64) TcGemmParams {
  CUtensorMap a_map[MAX_SEG];
  CUtensorMap b_map;
  CUtensorMap out_map[TC_MAX_OUT];
  CUtensorMap in_map[TC_MAX_IN];
  int nseg;
  int seg_nkb[MAX_SEG];
  int seg_shift[MAX_SEG];
  int seg_koff[MAX_SEG];
  int seg_shift_h[MAX_SEG];     // line shift of the segment (2-D WN taps)
  int seg_bcast[MAX_SEG];       // segment has no line dimension: its map has H = 1 and line coordinate 0
  int B, T, H, tiles_per_batch, n_tiles, total_tiles, N;  // tiles_per_batch: tiles per LINE
  int h0, nh;                   // line window [h0, h0 + nh) of every batch item (nh = H: all lines)
  uint32_t idesc;
  uint32_t desc_lbo, desc_sbo;  // >>4 encoded; overridable by the self test
  const int* row_len;           // GemmDesc::row_len
};

struct alignas(64) TcWgradParams {
  CUtensorMap a_map[TC_MAX_WG];
  CUtensorMap b_map[TC_MAX_WG];
  CUtensorMap out_map[TC_MAX_WG];  // fp32 partials [splits][M][N]
  int nprob;
  int M[TC_MAX_WG], N[TC_MAX_WG], shift[TC_MAX_WG], a_c0[TC_MAX_WG], b_c0[TC_MAX_WG];
  int shift_h[TC_MAX_WG], bcast[TC_MAX_WG];  // line shift / no-line flag of the B operand
  int tile_begin[TC_MAX_WG + 1];  // prefix sum of (m_tiles * n_tiles) per problem
  int n_tiles_n[TC_MAX_WG];
  // split-K over the flattened (batch, line, 64-row k-block) sequence: split s covers k-block units
  // [s * units_per_split, (s+1) * units_per_split) and accumulates ACROSS lines / batch items in TMEM
  int B, T, H, units_per_batch, total_units, units_per_split, splits, total_work;  // units_per_batch: per LINE
  uint32_t idesc;
  uint32_t desc_lbo, desc_sbo;
};

// ------------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// arrive on the barrier at shared::cluster address `addr` (possibly in the peer CTA)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(addr) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t addr = smem_u32(bar);
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}" ::"r"(addr),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// shared::cluster address of the same variable in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// TMA loads; `bar` is a shared::cluster mbarrier address (cta_group::2: it may live in the peer CTA)
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// slab operand tile: coordinates (channel, time, line, batch)
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
          dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_local(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1,
                                                  int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
          dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
// CTA-local TMA load (epilogue inputs)
__device__ __forceinline__ void tma_load_3d_local(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1,
                                                  int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// TMA store shared -> global (bulk async-group completion)
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(src), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// completion of all prior tcgen05.mma of this thread -> arrive on the barrier at this offset in BOTH CTAs
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"((uint16_t)3)
      : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread = one accumulator row)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n\t"
      "tcgen05.wait::ld.sync.aligned;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// 32 lanes x 16 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n\t"
      "tcgen05.wait::ld.sync.aligned;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// UMMA shared-memory descriptor (sm_100 "version 1"), SWIZZLE_128B
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_enc, uint32_t sbo_enc) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)(lbo_enc & 0x3FFF) << 16;
  d |= (uint64_t)(sbo_enc & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;  // SWIZZLE_128B
  return d;
}

// instruction descriptor for kind::f16, fp32 accumulate
inline uint32_t make_idesc(int is_fp16, int M, int N, int a_mn_major, int b_mn_major) {
  uint32_t fmt = is_fp16 ? 0u : 1u;  // 0 = F16, 1 = BF16
  uint32_t d = 0;
  d |= 1u << 4;                      // D format F32
  d |= fmt << 7;                     // A format
  d |= fmt << 10;                    // B format
  d |= (uint32_t)(a_mn_major & 1) << 15;
  d |= (uint32_t)(b_mn_major & 1) << 16;
  d |= (uint32_t)(N >> 3) << 17;
  d |= (uint32_t)(M >> 4) << 24;
  return d;
}

// ------------------------------------------------------------------------------------------------
// epilogue staging: one 32-row x 32-column chunk per warp, thread `lane` owns row `lane`.
//   16-bit chunk: 32 x 64 B,  TMA SWIZZLE_64B  (16-byte slot j of row r lives at slot j ^ ((r >> 1) & 3))
//   fp32 chunk:   32 x 128 B, TMA SWIZZLE_128B (16-byte slot j of row r lives at slot j ^ (r & 7))
// Both are bank-conflict free for the row-per-thread 16-byte accesses of a quarter warp.
// ------------------------------------------------------------------------------------------------
constexpr int TC_CHUNK16_BYTES = 32 * 64;
constexpr int TC_CHUNK32_BYTES = 32 * 128;

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void ld_shared_v4(uint32_t addr, uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(addr) : "memory");
}
// half h (0/1) of a 16-bit chunk row: 16 columns = two 16-byte slots (2h, 2h+1)
__device__ __forceinline__ void stage_store16h(uint32_t buf, int lane, int h, const uint32_t (&o)[8]) {
  const uint32_t base = buf + lane * 64;
  const int sw = (lane >> 1) & 3;
#pragma unroll
  for (int j = 0; j < 2; ++j)
    st_shared_v4(base + (((2 * h + j) ^ sw) << 4), o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
}
__device__ __forceinline__ void stage_load16(uint32_t buf, int lane, uint32_t (&o)[16]) {
  const uint32_t base = buf + lane * 64;
  const int sw = (lane >> 1) & 3;
#pragma unroll
  for (int j = 0; j < 4; ++j) ld_shared_v4(base + ((j ^ sw) << 4), o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
}
// half h of an fp32 chunk row: 16 columns = four 16-byte slots (4h .. 4h+3)
__device__ __forceinline__ void stage_store32h(uint32_t buf, int lane, int h, const uint32_t (&o)[16]) {
  const uint32_t base = buf + lane * 128;
  const int sw = lane & 7;
#pragma unroll
  for (int j = 0; j < 4; ++j)
    st_shared_v4(base + (((4 * h + j) ^ sw) << 4), o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
}

template <class Epi>
struct TcEpiTraits {
  static constexpr int kOutChunk = Epi::kOutF32 ? TC_CHUNK32_BYTES : TC_CHUNK16_BYTES;
  static constexpr int kOutBytes = Epi::kOutBufs * Epi::kOut * kOutChunk;
  static constexpr int kInBytes = Epi::kIn * TC_CHUNK16_BYTES;  // inputs: 16-bit, one chunk (re-armed as soon as it is read)
  static constexpr int kWarpBytes = kOutBytes + kInBytes;
  // column groups = draining warps per TMEM lane quadrant (fewer groups = less staging = more operand stages)
  template <int GW>
  static constexpr int ncg() { return (GW / 32) < Epi::kColGroups ? (GW / 32) : Epi::kColGroups; }
};

constexpr int TC_BAR_BYTES = 512;  // mbarriers + TMEM pointer

template <int BN, class Epi>
constexpr int tc_stage_bytes() { return TC_A_BYTES + (BN / 2) * 128; }
template <int BN, class Epi>
constexpr int tc_epi_bytes() {
  return 4 * TcEpiTraits<Epi>::template ncg<(Epi::kPaired ? BN / 2 : BN)>() * TcEpiTraits<Epi>::kWarpBytes;
}
template <int BN, class Epi>
constexpr int tc_num_stages() {
  int avail = TC_SMEM_LIMIT - 1024 - TC_BAR_BYTES - tc_epi_bytes<BN, Epi>();
  int s = avail / tc_stage_bytes<BN, Epi>();
  return s > 8 ? 8 : s;
}
template <int BN, class Epi>
constexpr size_t tc_smem_bytes() {
  return (size_t)tc_num_stages<BN, Epi>() * tc_stage_bytes<BN, Epi>() + tc_epi_bytes<BN, Epi>() + TC_BAR_BYTES + 1024;
}

struct TcSmem {
  uint8_t* stages;
  uint8_t* epi;        // TC_EPI_WARPS x per-warp staging (1 KB aligned)
  uint64_t* full;      // [STAGES]   (leader's is the one in use)
  uint64_t* empty;     // [STAGES]
  uint64_t* tmem_full; // [2]
  uint64_t* tmem_empty;// [2]        (leader's is the one in use)
  uint64_t* in_bar;    // [TC_EPI_WARPS] epilogue input loads
  uint32_t* tmem_ptr;
};

template <int STAGES>
__device__ __forceinline__ TcSmem tc_carve(uint8_t* raw, int stage_bytes, int epi_bytes) {
  static_assert((2 * STAGES + 4 + TC_EPI_WARPS) * 8 + 8 <= TC_BAR_BYTES, "barrier area too small");
  TcSmem s;
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~(uintptr_t)1023);
  s.stages = base;
  s.epi = base + STAGES * stage_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s.epi + epi_bytes);
  s.full = bars;
  s.empty = bars + STAGES;
  s.tmem_full = bars + 2 * STAGES;
  s.tmem_empty = bars + 2 * STAGES + 2;
  s.in_bar = bars + 2 * STAGES + 4;
  s.tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4 + TC_EPI_WARPS);
  return s;
}

// `drain_warps`: epilogue warps per CTA that drain accumulators (arrivals on the leader's tmem_empty per CTA)
template <int STAGES>
__device__ __forceinline__ void tc_setup(const TcSmem& s, int warp, int lane, int tmem_cols, int drain_warps) {
  if (warp == 1) {
    if (lane == 0) {
      for (int i = 0; i < STAGES; ++i) { mbar_init(&s.full[i], 1); mbar_init(&s.empty[i], 1); }
      for (int i = 0; i < 2; ++i) { mbar_init(&s.tmem_full[i], 1); mbar_init(&s.tmem_empty[i], 2 * drain_warps); }
      for (int i = 0; i < TC_EPI_WARPS; ++i) mbar_init(&s.in_bar[i], 1);
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc(s.tmem_ptr, tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  cluster_sync_all();  // both CTAs: barriers initialised, TMEM allocated
  tc_fence_after();
}

__device__ __forceinline__ void tc_teardown(uint32_t tmem_base, int warp, int tmem_cols) {
  tc_fence_before();
  __syncwarp();
  cluster_sync_all();  // every MMA, remote arrive and TMEM read of the pair has finished
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// ------------------------------------------------------------------------------------------------
// K-major GEMM with fused epilogue
// ------------------------------------------------------------------------------------------------
template <int BN, class Epi>
__global__ void __launch_bounds__(TC_THREADS, 1) tc_gemm_kernel(const __grid_constant__ TcGemmParams p, const Epi epi) {
  extern __shared__ uint8_t smem_raw[];
  constexpr int STAGES = tc_num_stages<BN, Epi>();
  constexpr int STAGE_BYTES = tc_stage_bytes<BN, Epi>();
  using ET = TcEpiTraits<Epi>;
  static_assert(STAGES >= 2, "epilogue staging leaves no room for the operand pipeline");
  const TcSmem s = tc_carve<STAGES>(smem_raw, STAGE_BYTES, tc_epi_bytes<BN, Epi>());
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < p.nseg; ++i) prefetch_tmap(&p.a_map[i]);
    prefetch_tmap(&p.b_map);
    for (int i = 0; i < Epi::kOut; ++i) prefetch_tmap(&p.out_map[i]);
    for (int i = 0; i < Epi::kIn; ++i) prefetch_tmap(&p.in_map[i]);
  }
  constexpr int GW = Epi::kPaired ? BN / 2 : BN;   // epilogue columns of one tile (gate channels when paired)
  constexpr int NCG = ET::template ncg<GW>();       // column groups = draining warps per TMEM lane quadrant
  constexpr int NCH = GW / (32 * NCG);             // 32-column chunks per warp per tile
  pdl_trigger();  // the next kernel of the stream may set itself up while this one runs
  tc_setup<STAGES>(s, warp, lane, 2 * BN, 4 * NCG);
  const uint32_t tmem_base = *s.tmem_ptr;
  pdl_wait();     // everything above touched no global memory; the predecessor's results are visible from here on

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = pair; tile < p.total_tiles; tile += npairs) {
        int nt = tile % p.n_tiles, rt = tile / p.n_tiles;
        int line = rt / p.tiles_per_batch, t0 = (rt % p.tiles_per_batch) * (2 * TC_BM) + rank * TC_BM;
        int b = line / p.nh, h = p.h0 + (line - b * p.nh);
        int n0 = nt * BN + rank * (BN / 2);
        for (int sg = 0; sg < p.nseg; ++sg) {
          const int hs = p.seg_bcast[sg] ? 0 : h + p.seg_shift_h[sg];
          for (int kb = 0; kb < p.seg_nkb[sg]; ++kb) {
            mbar_wait(&s.empty[stage], phase ^ 1);
            uint32_t sa = smem_u32(s.stages + stage * STAGE_BYTES);
            if (rank == 0) mbar_arrive_expect_tx(&s.full[stage], 2 * STAGE_BYTES);
            uint32_t bar = mapa_shared(smem_u32(&s.full[stage]), 0);
            tma_load_4d(sa, &p.a_map[sg], bar, kb * TC_BK, t0 + p.seg_shift[sg], hs, b);
            tma_load_2d(sa + TC_A_BYTES, &p.b_map, bar, p.seg_koff[sg] + kb * TC_BK, n0);
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      int total_kb = 0;
      for (int sg = 0; sg < p.nseg; ++sg) total_kb += p.seg_nkb[sg];
      for (int tile = pair; tile < p.total_tiles; tile += npairs) {
        mbar_wait(&s.tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < total_kb; ++kb) {
          mbar_wait(&s.full[stage], phase);
          tc_fence_after();
          uint32_t sa = smem_u32(s.stages + stage * STAGE_BYTES);
          uint64_t adesc = make_smem_desc(sa, p.desc_lbo, p.desc_sbo);
          uint64_t bdesc = make_smem_desc(sa + TC_A_BYTES, p.desc_lbo, p.desc_sbo);
#pragma unroll
          for (int k = 0; k < TC_BK / 16; ++k) {
            // +32 bytes (>>4 = 2) per K=16 step inside the 128B swizzle row
            umma_f16(d_tmem, adesc + 2 * k, bdesc + 2 * k, p.idesc, (kb > 0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&s.empty[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&s.tmem_full[acc]);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else if ((warp - 2) >> 2 < NCG) {
    const int e = warp - 2;
    const int q = warp & 3;          // TMEM lane quadrant this warp may access (hardware: warp id % 4)
    const int cg = e >> 2;           // column group of this warp
    constexpr int OUTW = Epi::kOutF32 ? 16 : 8;  // registers per 16-column output fragment
    const uint32_t wbuf = smem_u32(s.epi + e * ET::kWarpBytes);
    const uint32_t ibuf = wbuf + ET::kOutBytes;
    uint64_t* ibar = s.in_bar + e;
    const uint32_t tmem_empty_addr = mapa_shared(smem_u32(&s.tmem_empty[0]), 0);
    int acc = 0;
    uint32_t acc_phase = 0;
    int ob = 0;        // output staging buffer in use
    uint32_t it = 0;   // running chunk counter (phase of the input barrier)

    // coordinates of chunk k of a tile: batch, line, first row of this warp, first epilogue column
    auto coords = [&](int tile, int k, int& b, int& h, int& r0, int& c0) {
      int nt = tile % p.n_tiles, rt = tile / p.n_tiles;
      int line = rt / p.tiles_per_batch;
      b = line / p.nh;
      h = p.h0 + (line - b * p.nh);
      r0 = (rt % p.tiles_per_batch) * (2 * TC_BM) + rank * TC_BM + q * 32;
      c0 = nt * GW + cg * (GW / NCG) + 32 * k;
    };
    auto issue_inputs = [&](int tile, int k) {
      if constexpr (Epi::kIn > 0) {
        if (lane == 0) {
          int b, h, r0, c0;
          coords(tile, k, b, h, r0, c0);
          fence_proxy_async();
          mbar_arrive_expect_tx(ibar, Epi::kIn * TC_CHUNK16_BYTES);
#pragma unroll
          for (int i = 0; i < Epi::kIn; ++i)
            tma_load_4d_local(ibuf + i * TC_CHUNK16_BYTES, &p.in_map[i], smem_u32(ibar), epi.in_col(i, c0), r0, h, b);
        }
      }
    };
    if (pair < p.total_tiles) issue_inputs(pair, 0);

    for (int tile = pair; tile < p.total_tiles; tile += npairs) {
      const uint32_t taddr = tmem_base + acc * BN + ((uint32_t)(q * 32) << 16) + cg * (GW / NCG);
      mbar_wait(&s.tmem_full[acc], acc_phase);
      tc_fence_after();
#pragma unroll 1
      for (int k = 0; k < NCH; ++k, ++it) {
        int b, h, r0, c0;
        coords(tile, k, b, h, r0, c0);
        // epilogue inputs: take this chunk into registers, then re-arm the buffer with the next chunk
        uint32_t in[Epi::kIn > 0 ? Epi::kIn : 1][16];
        if constexpr (Epi::kIn > 0) {
          mbar_wait(ibar, it & 1);
#pragma unroll
          for (int i = 0; i < Epi::kIn; ++i) stage_load16(ibuf + i * TC_CHUNK16_BYTES, lane, in[i]);
          __syncwarp();
          if (k + 1 < NCH) issue_inputs(tile, k + 1);
          else if (tile + npairs < p.total_tiles) issue_inputs(tile + npairs, 0);
        }
        // staging buffer `ob` must have been read by the TMA store issued Epi::kOutBufs chunks ago
        if (lane == 0) bulk_wait_read<Epi::kOutBufs - 1>();
        __syncwarp();
        const uint32_t obuf = wbuf + ob * Epi::kOut * ET::kOutChunk;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float v[16];
          uint32_t o[Epi::kOut][OUTW];
          tmem_ld16(taddr + 32 * k + 16 * h, v);
          if constexpr (Epi::kPaired) {
            float w[16];
            tmem_ld16(taddr + GW + 32 * k + 16 * h, w);
            if (h == 1 && k == NCH - 1) {  // TMEM buffer drained: hand it back to the MMA issuer
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive_cluster(tmem_empty_addr + 8 * acc);
            }
            epi.compute(c0 + 16 * h, v, w, o);
          } else {
            if (h == 1 && k == NCH - 1) {
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive_cluster(tmem_empty_addr + 8 * acc);
            }
            if constexpr (Epi::kIn > 0) {
              uint32_t inh[Epi::kIn][8];
#pragma unroll
              for (int i = 0; i < Epi::kIn; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) inh[i][j] = in[i][8 * h + j];
              epi.compute(c0 + 16 * h, v, inh, o);
            } else {
              epi.compute(c0 + 16 * h, v, o);
            }
          }
          if (p.row_len != nullptr && r0 + lane >= __ldg(p.row_len + b)) {   // past the item's end: select 0
#pragma unroll
            for (int i = 0; i < Epi::kOut; ++i)
#pragma unroll
              for (int j = 0; j < OUTW; ++j) o[i][j] = 0u;
          }
#pragma unroll
          for (int i = 0; i < Epi::kOut; ++i) {
            if constexpr (Epi::kOutF32) stage_store32h(obuf + i * ET::kOutChunk, lane, h, o[i]);
            else stage_store16h(obuf + i * ET::kOutChunk, lane, h, o[i]);
          }
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
#pragma unroll
          for (int i = 0; i < Epi::kOut; ++i)
            tma_store_4d(&p.out_map[i], obuf + i * ET::kOutChunk, epi.out_col(i, c0), r0, h, b);
          bulk_commit();
        }
        if (Epi::kOutBufs > 1) ob ^= 1;
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (lane == 0) bulk_wait_read<0>();  // staging must outlive the last stores' reads
  }
  tc_teardown(tmem_base, warp, 2 * BN);
}

// ------------------------------------------------------------------------------------------------
// MN-major weight-gradient GEMM: D[m][n] = sum_t A[t][m] * B[t+shift][n], split over time chunks.
// The pair computes a 256 (m) x BN (n) tile: each CTA loads its 128 m-columns of A and its BN/2
// n-columns of B; fp32 partial tiles leave through the TMA store path.
// ------------------------------------------------------------------------------------------------
struct WgradEpiShape {  // staging shape of the weight-gradient epilogue (fp32, one stream)
  static constexpr bool kOutF32 = true, kPaired = false;
  static constexpr int kOut = 1, kIn = 0, kOutBufs = 1, kColGroups = 4;
};

template <int BN>
__global__ void __launch_bounds__(TC_THREADS, 1) tc_wgrad_kernel(const __grid_constant__ TcWgradParams p) {
  extern __shared__ uint8_t smem_raw[];
  constexpr int STAGES = tc_num_stages<BN, WgradEpiShape>();
  constexpr int STAGE_BYTES = tc_stage_bytes<BN, WgradEpiShape>();
  using ET = TcEpiTraits<WgradEpiShape>;
  constexpr int BOX_BYTES = 64 * 128;  // {64 channels, 64 time rows} x 16 bit
  const TcSmem s = tc_carve<STAGES>(smem_raw, STAGE_BYTES, tc_epi_bytes<BN, WgradEpiShape>());
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  if (warp == 0 && lane == 0) {
    for (int i = 0; i < p.nprob; ++i) { prefetch_tmap(&p.a_map[i]); prefetch_tmap(&p.b_map[i]); prefetch_tmap(&p.out_map[i]); }
  }
  constexpr int NCG = ET::template ncg<BN>();
  constexpr int NCH = BN / (32 * NCG);
  pdl_trigger();
  tc_setup<STAGES>(s, warp, lane, 2 * BN, 4 * NCG);
  const uint32_t tmem_base = *s.tmem_ptr;
  pdl_wait();
  const int tiles_total = p.tile_begin[p.nprob];

  // work item -> (problem, m tile, n tile, split); tiles vary fastest so that one time chunk of the
  // operands is reused from L2 by neighbouring CTAs
  auto decode = [&](int w, int& pr, int& m0, int& n0, int& split) {
    split = w / tiles_total;
    int tl = w % tiles_total;
    pr = 0;
    while (tl >= p.tile_begin[pr + 1]) ++pr;
    tl -= p.tile_begin[pr];
    m0 = (tl / p.n_tiles_n[pr]) * (2 * TC_BM);
    n0 = (tl % p.n_tiles_n[pr]) * BN;
  };

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int w = pair; w < p.total_work; w += npairs) {
        int pr, m0, n0, split;
        decode(w, pr, m0, n0, split);
        const int u0 = split * p.units_per_split, u1 = min(u0 + p.units_per_split, p.total_units);
        const int ma = p.a_c0[pr] + m0 + rank * TC_BM;
        const int nb = p.b_c0[pr] + n0 + rank * (BN / 2);
        int line = u0 / p.units_per_batch, t = (u0 - line * p.units_per_batch) * TC_BK;
        int b = line / p.H, h = line - b * p.H;
        const int dh = p.shift_h[pr], bc = p.bcast[pr];
        for (int u = u0; u < u1; ++u) {
          mbar_wait(&s.empty[stage], phase ^ 1);
          uint32_t sa = smem_u32(s.stages + stage * STAGE_BYTES);
          if (rank == 0) mbar_arrive_expect_tx(&s.full[stage], 2 * STAGE_BYTES);
          uint32_t bar = mapa_shared(smem_u32(&s.full[stage]), 0);
#pragma unroll
          for (int j = 0; j < TC_BM / 64; ++j) tma_load_4d(sa + j * BOX_BYTES, &p.a_map[pr], bar, ma + j * 64, t, h, b);
#pragma unroll
          for (int j = 0; j < BN / 128; ++j)
            tma_load_4d(sa + TC_A_BYTES + j * BOX_BYTES, &p.b_map[pr], bar, nb + j * 64, t + p.shift[pr],
                        bc ? 0 : h + dh, b);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
          t += TC_BK;
          if (t >= p.units_per_batch * TC_BK) {
            t = 0;
            if (++h == p.H) { h = 0; ++b; }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int w = pair; w < p.total_work; w += npairs) {
        int pr, m0, n0, split;
        decode(w, pr, m0, n0, split);
        const int nkb = min(p.units_per_split, p.total_units - split * p.units_per_split);
        mbar_wait(&s.tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&s.full[stage], phase);
          tc_fence_after();
          uint32_t sa = smem_u32(s.stages + stage * STAGE_BYTES);
          uint64_t adesc = make_smem_desc(sa, p.desc_lbo, p.desc_sbo);
          uint64_t bdesc = make_smem_desc(sa + TC_A_BYTES, p.desc_lbo, p.desc_sbo);
#pragma unroll
          for (int k = 0; k < TC_BK / 16; ++k) {
            // 16 time rows x 128 B = 2048 B (>>4 = 128) per K=16 step
            umma_f16(d_tmem, adesc + 128 * k, bdesc + 128 * k, p.idesc, (kb > 0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&s.empty[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&s.tmem_full[acc]);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else if ((warp - 2) >> 2 < NCG) {
    const int e = warp - 2;
    const int q = warp & 3;
    const int cg = e >> 2;
    const uint32_t wbuf = smem_u32(s.epi + e * ET::kWarpBytes);
    const uint32_t tmem_empty_addr = mapa_shared(smem_u32(&s.tmem_empty[0]), 0);
    int acc = 0;
    uint32_t acc_phase = 0;
    int ob = 0;
    for (int w = pair; w < p.total_work; w += npairs) {
      int pr, m0, n0, split;
      decode(w, pr, m0, n0, split);
      mbar_wait(&s.tmem_full[acc], acc_phase);
      tc_fence_after();
      const int mq = m0 + rank * TC_BM + q * 32;
      const uint32_t taddr = tmem_base + acc * BN + ((uint32_t)(q * 32) << 16) + cg * (BN / NCG);
#pragma unroll 1
      for (int k = 0; k < NCH; ++k) {
        if (lane == 0) bulk_wait_read<WgradEpiShape::kOutBufs - 1>();
        __syncwarp();
        const uint32_t obuf = wbuf + ob * TC_CHUNK32_BYTES;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float v[16];
          tmem_ld16(taddr + 32 * k + 16 * h, v);
          if (h == 1 && k == NCH - 1) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(tmem_empty_addr + 8 * acc);
          }
          uint32_t o[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) o[j] = __float_as_uint(v[j]);
          stage_store32h(obuf, lane, h, o);
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          tma_store_4d(&p.out_map[pr], obuf, n0 + cg * (BN / NCG) + 32 * k, mq, 0, split);
          bulk_commit();
        }
        if (WgradEpiShape::kOutBufs > 1) ob ^= 1;
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (lane == 0) bulk_wait_read<0>();
  }
  tc_teardown(tmem_base, warp, 2 * BN);
}

// ------------------------------------------------------------------------------------------------
// host side: tensor maps + launches
// ------------------------------------------------------------------------------------------------
enum TcMapKind {
  TC_MAP_OPERAND = 0,   // 16-bit, 128B swizzle (UMMA operand tiles)
  TC_MAP_CHUNK16 = 1,   // 16-bit, 64B swizzle, box {32, 32, 1} (epilogue streams)
  TC_MAP_CHUNK32 = 2,   // fp32,   128B swizzle, box {32, 32, 1}
};
// cached tensor map over a slab [B][H][T][ld] of which the first C channels are valid (dims (C, T, H, B));
// box (box_c, box_t, 1, 1); zero OOB fill
int get_slab_map(CUtensorMap* m, const void* ptr, int C, int ld, int T, int H, int B, int box_c, int box_t,
                 int is_fp16, int kind);
// 16-bit tensor map over a matrix [rows][ld]: dims (ld, rows), box (64, box_rows)
int get_matrix_map(CUtensorMap* m, const void* ptr, int ld, int rows, int box_rows, int is_fp16);
int tc_launch_pairs(const void* kern, size_t smem, int pairs, void** args, cudaStream_t st, int threads = TC_THREADS);
int tc_launch_pairs_coresident(const void* kern, size_t smem, int pairs, void** args, cudaStream_t st,
                               int threads = TC_THREADS);

template <int BN, class Epi>
int tc_gemm_launch_bn(const GemmDesc& d, const TcIo& io, const Epi& epi, cudaStream_t st, int lbo_override = -1,
                      int sbo_override = -1) {
  TcGemmParams p;
  memset(&p, 0, sizeof(p));
  p.nseg = d.nseg;
  const int H = d.H > 0 ? d.H : 1;
  for (int s = 0; s < d.nseg; ++s) {
    CMWG_REQUIRE(d.seg[s].K % TC_BK == 0, "tc_gemm: segment K=%d not a multiple of %d", d.seg[s].K, TC_BK);
    CMWG_PROPAGATE(get_slab_map(&p.a_map[s], d.seg[s].a, d.seg[s].lda, d.seg[s].lda, d.T, d.seg[s].bcast_h ? 1 : H, d.B,
                                TC_BK, TC_BM, d.is_fp16, TC_MAP_OPERAND));
    p.seg_nkb[s] = d.seg[s].K / TC_BK;
    p.seg_shift[s] = d.seg[s].shift;
    p.seg_koff[s] = d.seg[s].koff;
    p.seg_shift_h[s] = d.seg[s].shift_h;
    p.seg_bcast[s] = d.seg[s].bcast_h;
  }
  CMWG_PROPAGATE(get_matrix_map(&p.b_map, d.w, d.ldw, d.n_rows_w, BN / 2, d.is_fp16));
  for (int i = 0; i < Epi::kOut; ++i) {
    CMWG_REQUIRE(io.out[i].ptr != nullptr && (io.out[i].is_f32 != 0) == Epi::kOutF32, "tc_gemm: output stream %d mismatch", i);
    CMWG_PROPAGATE(get_slab_map(&p.out_map[i], io.out[i].ptr, io.out[i].cols, io.out[i].ld, d.T, H, d.B, 32, 32, d.is_fp16,
                                Epi::kOutF32 ? TC_MAP_CHUNK32 : TC_MAP_CHUNK16));
  }
  for (int i = 0; i < Epi::kIn; ++i) {
    CMWG_REQUIRE(io.in[i].ptr != nullptr && !io.in[i].is_f32, "tc_gemm: input stream %d mismatch", i);
    CMWG_PROPAGATE(get_slab_map(&p.in_map[i], io.in[i].ptr, io.in[i].cols, io.in[i].ld, d.T, H, d.B, 32, 32, d.is_fp16,
                                TC_MAP_CHUNK16));
  }
  p.B = d.B; p.T = d.T; p.H = H; p.N = d.N;
  p.tiles_per_batch = ceil_div(d.T, 2 * TC_BM);
  p.n_tiles = ceil_div(d.N, BN);
  p.h0 = d.nh > 0 ? d.h0 : 0;
  p.nh = d.nh > 0 ? d.nh : H;
  CMWG_REQUIRE(p.h0 >= 0 && p.h0 + p.nh <= H, "tc_gemm: line window [%d, %d) outside [0, %d)", p.h0, p.h0 + p.nh, H);
  p.total_tiles = d.B * p.nh * p.tiles_per_batch * p.n_tiles;
  p.idesc = make_idesc(d.is_fp16, 2 * TC_BM, BN, 0, 0);
  p.desc_lbo = lbo_override >= 0 ? (uint32_t)lbo_override : 1u;
  p.desc_sbo = sbo_override >= 0 ? (uint32_t)sbo_override : (1024u >> 4);
  CMWG_REQUIRE(d.row_len == nullptr || H == 1, "tc_gemm: per-item lengths need the 1-D layout");
  p.row_len = d.row_len;
  if (p.total_tiles == 0) return CMWG_OK;
  auto kern = tc_gemm_kernel<BN, Epi>;
  constexpr size_t smem = tc_smem_bytes<BN, Epi>();
  static_assert(smem <= TC_SMEM_LIMIT, "shared memory budget exceeded");
  static bool attr_set = false;
  if (!attr_set) {
    CMWG_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set = true;
  }
  int pairs = std::min(p.total_tiles, num_sms() / 2);
  ProfScope prof(st, d.tag);
  void* args[2] = {(void*)&p, (void*)&epi};
  CMWG_PROPAGATE(tc_launch_pairs((const void*)kern, smem, pairs, args, st));
  CMWG_COUNT_LAUNCH();
  return CMWG_OK;
}

template <class Epi>
int tc_gemm_launch(const GemmDesc& d, const TcIo& io, const Epi& epi, cudaStream_t st) {
  if (d.bn == 256) return tc_gemm_launch_bn<256, Epi>(d, io, epi, st);
  return tc_gemm_launch_bn<128, Epi>(d, io, epi, st);
}

// Split-K plan of the weight-gradient launches: problems are grouped by N tile width (>= 256 / < 256) and
// every group gets as many splits as fit one wave of CTA pairs.  splits_out[i] = splits of problem i
// (its partial buffer must hold splits_out[i] * M * N floats).  force_splits > 0 overrides the plan.
// B counts LINES here (batch items x lines per item); H only tells the kernel how lines group into batch items.
void tc_wgrad_plan(const WgradProblem* probs, int nprob, int B, int H, int T, int force_splits, int* splits_out);
int tc_wgrad_launch(const WgradProblem* probs, int nprob, int B, int H, int T, int is_fp16, cudaStream_t st,
                    int force_splits = 0, int lbo_override = -1, int sbo_override = -1);

}  // namespace cmwg
