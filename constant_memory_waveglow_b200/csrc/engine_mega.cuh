// Whole-WN forward as ONE persistent tcgen05 kernel (1-D WN, 16-bit operands).
//
// The layer-at-a-time pipeline of wn_pipeline.cu launches 2 GEMMs per layer; every launch boundary is a device-wide
// barrier that costs a pipeline fill + drain (~8 us measured at the LJ shapes) and rounds the tile count up to whole
// waves of 74 CTA pairs (384 gate tiles = 5.19 waves -> 6).  Here every GEMM tile of every layer is a TASK in one
// global, topologically ordered list
//     for layer i:  G(i, rt, nt)  gate GEMM tiles (dilated conv + conditioning, tanh*sigmoid epilogue)
//                   R(i, rt)      residual GEMM tiles (W_o[:Cr], epilogue adds the (hi, lo) pair of the layer input)
//     then          S(rt)         skip GEMM tiles (all layers' W_o[Cr:], K-concatenated)
// (interleaved: slot u = layer * RT + rt holds G(u, *) and R(u - LAG), so a pair alternates MMA-heavy gate tiles with
// epilogue-heavy residual tiles and the residual epilogue drains one TMEM buffer while the next gate tile fills the other)
// and CTA pair p runs tasks p, p + P, p + 2P, ... (P pairs, all co-resident).  Dependencies are per ROW TILE, not per
// layer: R(i, rt) needs G(i, rt, *); G(i, rt, *) needs R(i-1, rt-1 .. rt+1) (the dilated taps reach at most one
// 256-row tile away); S(rt) needs G(depth-1, rt, *).  They are tracked by counters in global memory: every epilogue warp
// adds 1 (release) to its task's counter once its TMA stores have COMPLETED, and the TMA producer (and, for R, the
// epilogue's input loader) polls (acquire) before it issues loads.  The list is in dependency order and a pair executes
// its tasks in list order, so the lowest unfinished task is always runnable: no deadlock as long as all pairs are
// resident (grid <= SM count / 2, one CTA per SM).  A wait that exceeds ~2 s traps instead of hanging the device.
//
// Roles, rings, TMEM double buffering and the epilogue functors are those of engine_tc.cuh; the epilogue switches
// functor per task (warp-uniform), the residual epilogue works IN PLACE in its staging buffers (inputs are read into
// registers, outputs overwrite them) and a third output stream waits in registers for the first two stores, so 4 KB of
// staging per warp suffice and five operand stages fit.
#pragma once
#include "engine_tc.cuh"
#include "epilogues_tc.cuh"

namespace cmwg {

constexpr int MEGA_D = 8;        // layers
// Warp 18 is a SECOND TMA producer.  One thread issuing both operand loads of every k-block spends ~590 cycles per k-block
// on its own instruction stream (barrier wait, expect_tx, two UTMALDG, task decode, dependency polling: measured with
// CMWG_MEGA_CLK), MORE than the 512 cycles the tensor pipe needs for the k-block -- the MMA issuer waited 27 % of the kernel
// on operands.  The weight (B) tiles depend on nothing, so a second thread streams them: it walks the same task list and
// waits only for free ring slots, while warp 0 keeps the activation (A) tiles and the dependency counters.
// Warp 19 is a SCOUT.  Checking a task's dependency counters costs an L2 round trip plus an acquire fence (~1200 cycles with
// the proxy fence) even when they were satisfied long ago; done by the producer between two tasks, that gap -- and the TMA
// latency behind it -- is longer than the 4 k-blocks of work the ring holds, so the tensor pipe ran dry at every task
// boundary.  The scout walks the task list ahead of the producer, does the waiting, and publishes "tasks cleared" in shared
// memory; the producer's check is then a shared-memory load.
constexpr int MEGA_THREADS = TC_THREADS + 64;
constexpr int MEGA_BWARP = TC_THREADS / 32;       // index of the weight-producer warp
constexpr int MEGA_SWARP = TC_THREADS / 32 + 1;   // index of the scout warp

__device__ __forceinline__ void st_release_cta_u32(uint32_t* p, uint32_t v) {
  asm volatile("st.release.cta.shared::cta.u32 [%0], %1;" ::"r"(smem_u32(p)), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_cta_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.cta.shared::cta.u32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)) : "memory");
  return v;
}
// producer side: task number `n` (1-based count of this pair's non-empty tasks) has been cleared by the scout
__device__ __forceinline__ void mega_wait_cleared(const uint32_t* cleared, uint32_t n) {
  while (ld_acquire_cta_u32(cleared) < n) { }
  asm volatile("fence.proxy.async.global;" ::: "memory");
}
constexpr int MEGA_BN = 256;     // N tile of every task
enum { MEGA_G = 0, MEGA_R = 1, MEGA_S = 2, MEGA_NONE = 3 };

struct alignas(64) MegaParams {
  CUtensorMap hin_op[MEGA_D];   // operand maps (64 ch x 128 rows, 128B swizzle): layer inputs (hi halves)
  CUtensorMap g_op[MEGA_D];     // operand maps: gate outputs
  CUtensorMap cond_op;          // operand map: packed conditioning
  CUtensorMap pa[MEGA_D], pb[MEGA_D], ps;                       // weights (64 x 128-row boxes)
  CUtensorMap g_c16[MEGA_D], b_c16[MEGA_D];                     // 32 x 32 chunk maps: gate outputs, saved sigmoid
  CUtensorMap hi_c16[MEGA_D], lo_c16[MEGA_D];                   // chunk maps: (hi, lo) pair of every layer's INPUT
  CUtensorMap skip_c32;                                         // fp32 chunk map: cumulative skip
  uint32_t* flags;              // [depth][2][RT]: gate-done / residual-done counters (zeroed before the launch)
  int depth, B, T, tiles_per_batch, RT;
  int ngt;                      // gate N tiles
  int taps, kb_h, kb_c, kb_g;   // taps; k-blocks per tap / of the conditioning / of one gate output
  int kc_last;                  // K = 16 steps of the conditioning's last k-block that hold real channels (1 .. 4)
  // layer 0 with the start conv folded in (PackedLayout::PA0f / PB0f): its gate tiles read only the conditioning slab (whose
  // padding columns carry the taps of x_a), its residual tiles add one k-block of that slab (W_start x_a = h_0) to W_res g_0
  // and have nothing to load in their epilogue
  int fold0;
  int kc_last0;                 // as kc_last, counting the x_a columns too
  CUtensorMap pa0f, pb0f;
  int Cd, f16;
  uint32_t idesc, desc_lbo, desc_sbo;
  int lag;                      // residual tiles trail their gate tiles by `lag` row-tile slots (< RT - 1)
  int total_tasks;
  int lagged;                   // signal a unit's completion one unit later (its stores complete behind the next unit's work)
  long long* clk;               // nullptr, or [CTAs][18 warps][16] cycle accumulators (CMWG_MEGA_CLK: where the roles wait)
  int dbg;                      // timing experiments only (CMWG_MEGA_DBG): 1 no producer waits, 2 no signals, 4 no wait_all
  int dual;                     // 1: warp MEGA_BWARP issues the weight tiles (default), 0: warp 0 issues both operands
  // `end` conv fused into the skip tiles' epilogue (model/waveglow.py:92,105): lst[b][o][t] = sum_c w_end[o][c] * cum_skip[b][t][c].
  // lst == nullptr: off (the fp32 skip slab is written and a separate kernel reads it back).
  // Residual tiles with DIRECT global loads / stores of the (hi, lo) pairs (row-per-thread 32-byte vectors) instead of TMA
  // chunks through the staging buffers: the small epilogue transfers no longer queue behind the operand stream in the SM's
  // TMA unit (res_direct = 0: the TMA path).
  const uint16_t* hi_ptr[MEGA_D];   // layer inputs, hi halves  [rows][Cr]
  uint16_t* lo_ptr[MEGA_D];         // layer inputs, lo halves
  uint16_t* hi_out_ptr[MEGA_D];     // same slabs, writable view (hi_out_ptr[i] = hi_ptr[i])
  int res_direct;
  int res_lo;                   // 1: the residual stream is a (hi, lo) pair of 16-bit slabs; 0: the operand slab alone (AddTcEpi)
  int gate_mix;                 // GateTcEpi::mix
  float* lst;                   // (B, cout, T) fp32 NCL
  const float* w_end;           // [MEGA_END_MAXC][Cs] fp32, rows >= cout zero
  int cout;
  int store_skip;               // also keep the fp32 cumulative skip slab (training: the `end` weight gradient reads it)
  // Per-item lengths (cmwg_wn_forward_varlen).  rt_tab == nullptr: every item has tiles_per_batch row tiles and row tile rt is
  // (rt / tiles_per_batch, rt % tiles_per_batch).  Otherwise rt_tab[rt] = (item, tile within the item, tiles of the item): the
  // list holds only the tiles that contain valid rows.  row_len != nullptr: the residual epilogues write 0 at rows
  // t >= row_len[item], so every layer input is zero past the item's end, as the TMA zero fill leaves it for a call of that length.
  const int4* rt_tab;
  const int* row_len;
};

struct MegaTile {
  int b, tb, ntb;   // batch item, row tile within it, row tiles of the item
};
__host__ __device__ __forceinline__ MegaTile mega_tile(const int4* tab, int tiles_per_batch, int rt) {
  MegaTile m;
  if (tab != nullptr) {
    const int4 e = tab[rt];
    m.b = e.x; m.tb = e.y; m.ntb = e.z;
  } else {
    m.b = rt / tiles_per_batch; m.tb = rt - m.b * tiles_per_batch; m.ntb = tiles_per_batch;
  }
  return m;
}
// row `trow` of item b lies past the item's end: its residual output is 0 (a select: the accumulator there may be anything)
__device__ __forceinline__ bool mega_dead_row(const int* row_len, int b, int trow) {
  return row_len != nullptr && trow >= __ldg(row_len + b);
}

__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_add_u32(uint32_t* p, uint32_t v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// generic <-> async proxy ordering for GLOBAL memory only (flag observed by a generic load -> TMA loads of the data it guards;
// TMA stores completed -> generic release of the flag).  The unqualified form also covers shared memory and was measured to cost
// the producer ~700 cycles per task with five TMA stages in flight.
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async.global;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_complete() {  // all but the N most recent bulk groups of this thread are COMPLETE
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
// completion signal of one unit (one TMEM buffer's worth of epilogue) of one warp
struct MegaSig {
  uint32_t* flag;     // global dependency counter (nullptr: nothing depends on this unit)
  uint32_t cnt;       // shared-memory arrival counter of the CTA's epilogue warps for this unit
};
// One release per CTA and unit instead of one per warp: the warps count in shared memory (acq_rel, so the last arrival
// has observed the others' completed stores) and the 16th publishes all of them.
__device__ __forceinline__ void mega_signal(const MegaSig& sg) {
  if (sg.flag == nullptr) return;
  asm volatile("fence.proxy.async.global;" ::: "memory");
  uint32_t old;
  asm volatile("atom.acq_rel.cta.shared::cta.add.u32 %0, [%1], 1;" : "=r"(old) : "r"(sg.cnt) : "memory");
  if ((old & (TC_EPI_WARPS - 1)) == TC_EPI_WARPS - 1) red_release_add_u32(sg.flag, (uint32_t)TC_EPI_WARPS);
}

// ~20 s at 1.9 GHz.  A wait this long means a lost dependency (a bug) -- or that part of this grid is not resident because
// another kernel holds its SMs for that long; a collective that waits for a peer rank is the one legitimate case, and it is
// given time: the kernel reports which CTA gave up before it traps.
constexpr long long MEGA_WAIT_LIMIT = 40000000000ll;
__device__ __noinline__ void mega_timeout(const uint32_t* p, uint32_t target) {
  printf("cmwg_b200 task kernel: CTA %d waited > %lld cycles for dependency counter %p (value %u, needs %u); trapping\n",
         (int)blockIdx.x, MEGA_WAIT_LIMIT, (const void*)p, *(volatile const uint32_t*)p, target);
  __trap();
}
__device__ __forceinline__ void mega_wait_flag(const uint32_t* p, uint32_t target) {
  if (ld_acquire_u32(p) >= target) return;
  const long long t0 = clock64();
  while (ld_acquire_u32(p) < target) {
    __nanosleep(40);
    if (clock64() - t0 > MEGA_WAIT_LIMIT) mega_timeout(p, target);  // a lost dependency must not hang the device
  }
}

__device__ __forceinline__ uint32_t ld_relaxed_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// up to three counters polled with independent relaxed loads (one L2 round trip), then one acquire fence
__device__ __forceinline__ void mega_wait_flags3(const uint32_t* a, const uint32_t* b, const uint32_t* c, uint32_t target,
                                                 bool fence = true) {
  const long long t0 = clock64();
  while (true) {
    const uint32_t va = ld_relaxed_u32(a), vb = ld_relaxed_u32(b), vc = ld_relaxed_u32(c);
    if (va >= target && vb >= target && vc >= target) break;
    __nanosleep(40);
    if (clock64() - t0 > MEGA_WAIT_LIMIT) mega_timeout(b, target);
  }
  if (fence) asm volatile("fence.acq_rel.gpu;" ::: "memory");
}

struct MegaTask {
  int type, layer, rt, nt;
};
__host__ __device__ __forceinline__ MegaTask mega_decode(const MegaParams& p, int idx) {
  // slots 0 .. depth*RT + lag - 1, (ngt + 1) positions each: G(u = slot, nt) then R(u = slot - lag); positions whose
  // task does not exist are MEGA_NONE (skipped by every role alike); the skip tiles follow
  MegaTask t;
  const int per_slot = p.ngt + 1;
  const int slots = p.depth * p.RT + p.lag;
  t.nt = 0;
  if (idx >= slots * per_slot) {
    t.type = MEGA_S; t.layer = p.depth - 1; t.rt = idx - slots * per_slot;
    return t;
  }
  const int sl = idx / per_slot, w = idx - sl * per_slot;
  const int u = w < p.ngt ? sl : sl - p.lag;
  t.layer = u >= 0 ? u / p.RT : 0;
  t.rt = u - t.layer * p.RT;
  if (w < p.ngt) {
    t.type = u < p.depth * p.RT ? MEGA_G : MEGA_NONE;
    t.nt = w;
  } else {
    t.type = (u >= 0 && t.layer < p.depth - 1) ? MEGA_R : MEGA_NONE;
  }
  return t;
}
__device__ __forceinline__ uint32_t* mega_gflag(const MegaParams& p, int layer, int rt) {
  return p.flags + (size_t)(2 * layer) * p.RT + rt;
}
__device__ __forceinline__ uint32_t* mega_rflag(const MegaParams& p, int layer, int rt) {
  return p.flags + (size_t)(2 * layer + 1) * p.RT + rt;
}

// Epilogue of ONE task for one warp: GW epilogue columns per tile, four column groups (one per warp of the lane quadrant).
// kIn > 0: in-place staging -- chunk inputs are TMA-loaded into the buffers the outputs are later stored from; the
// caller has already issued chunk 0's inputs and made sure the staging buffers are free.  Immediate mode: ends with ALL
// of this warp's stores complete, then signals `flag`.  Lagged mode (`prev` != nullptr): waits only for the PREVIOUS unit's
// stores (which completed behind this unit's work), signals that unit and leaves this one pending in `prev`.
template <class Epi, int GW>
__device__ __forceinline__ void mega_epilogue_task(const Epi& epi, uint32_t tmem_tile, uint64_t* tmem_full, uint32_t full_phase,
                                                   uint32_t tmem_empty_remote, int q, int cg, int lane, uint32_t wbuf,
                                                   uint64_t* ibar, uint32_t& it, const CUtensorMap* om0,
                                                   const CUtensorMap* om1, const CUtensorMap* om2, const CUtensorMap* im0,
                                                   const CUtensorMap* im1, int b, int r0, int cbase, MegaSig sig, MegaSig* prev, int dbg, uint32_t* tt,
                                                   bool dead = false) {
  constexpr int NCH = GW / 128;                      // 32-column chunks per warp
  constexpr int OUTW = Epi::kOutF32 ? 16 : 8;
  constexpr int OCH = Epi::kOutF32 ? TC_CHUNK32_BYTES : TC_CHUNK16_BYTES;
  constexpr int NST = Epi::kOut < 2 ? Epi::kOut : 2;   // streams staged at once: the staging holds two 2 KB chunks, a third
                                                       // stream (saved sigmoid) waits in registers for the first stores
  const uint32_t taddr = tmem_tile + ((uint32_t)(q * 32) << 16) + cg * (GW / 4);
  const CUtensorMap* om[3] = {om0, om1, om2};
  const CUtensorMap* im[2] = {im0, im1};
  const uint32_t c_a = (uint32_t)clock();
  mbar_wait(tmem_full, full_phase);
  tc_fence_after();
  const uint32_t c_b = (uint32_t)clock();
#pragma unroll 1
  for (int k = 0; k < NCH; ++k) {
    const int c0 = cbase + cg * (GW / 4) + 32 * k;
    if (k > 0) {  // the previous chunk's stores must have read the staging buffers before they are overwritten
      if (lane == 0) {
        bulk_wait_read<0>();
        if constexpr (Epi::kIn > 0) {
          fence_proxy_async();
          mbar_arrive_expect_tx(ibar, Epi::kIn * TC_CHUNK16_BYTES);
#pragma unroll
          for (int i = 0; i < Epi::kIn; ++i)
            tma_load_4d_local(wbuf + i * TC_CHUNK16_BYTES, im[i], smem_u32(ibar), c0, r0, 0, b);
        }
      }
      __syncwarp();
    }
    uint32_t in[Epi::kIn > 0 ? Epi::kIn : 1][16];
    if constexpr (Epi::kIn > 0) {
      mbar_wait(ibar, it & 1);
      ++it;
#pragma unroll
      for (int i = 0; i < Epi::kIn; ++i) stage_load16(wbuf + i * TC_CHUNK16_BYTES, lane, in[i]);
      __syncwarp();
    }
    uint32_t keep[2][OUTW];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float v[16];
      uint32_t o[Epi::kOut][OUTW];
      tmem_ld16(taddr + 32 * k + 16 * h, v);
      if constexpr (Epi::kPaired) {
        float w[16];
        tmem_ld16(taddr + GW + 32 * k + 16 * h, w);
        if (h == 1 && k == NCH - 1) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(tmem_empty_remote);
        }
        epi.compute(c0 + 16 * h, v, w, o);
      } else {
        if (h == 1 && k == NCH - 1) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(tmem_empty_remote);
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
      if (dead) {   // this lane's row is past its item's end (per-item lengths)
#pragma unroll
        for (int i = 0; i < Epi::kOut; ++i)
#pragma unroll
          for (int j = 0; j < OUTW; ++j) o[i][j] = 0u;
      }
#pragma unroll
      for (int i = 0; i < NST; ++i) {
        if constexpr (Epi::kOutF32) stage_store32h(wbuf + i * OCH, lane, h, o[i]);
        else stage_store16h(wbuf + i * OCH, lane, h, o[i]);
      }
      if constexpr (Epi::kOut > 2) {
#pragma unroll
        for (int j = 0; j < OUTW; ++j) keep[h][j] = o[2][j];
      }
    }
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) {
#pragma unroll
      for (int i = 0; i < NST; ++i) tma_store_4d(om[i], wbuf + i * OCH, c0, r0, 0, b);
      bulk_commit();
    }
    if constexpr (Epi::kOut > 2 && !Epi::kOutF32) {
      if (lane == 0) bulk_wait_read<0>();
      __syncwarp();
      stage_store16h(wbuf, lane, 0, keep[0]);
      stage_store16h(wbuf, lane, 1, keep[1]);
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        tma_store_4d(om[2], wbuf, c0, r0, 0, b);
        bulk_commit();
      }
    }
  }
  const uint32_t c_c = (uint32_t)clock();
  if (lane == 0) {
    if (dbg & 2) sig.flag = nullptr;
    if (prev != nullptr) {
      bulk_wait_complete<NCH * (Epi::kOut > 2 ? 2 : 1)>();  // this unit's own groups may be pending, everything older is complete
      mega_signal(*prev);
      *prev = sig;
    } else {
      bulk_wait_all();            // stores COMPLETE (not just read): the results are in global memory
      mega_signal(sig);
    }
  }
  __syncwarp();
  tt[0] += c_b - c_a;            // waiting for the accumulator
  tt[1] += c_c - c_b;            // drain + functor + staging + store issue (+ input waits)
  tt[2] += (uint32_t)clock() - c_c;  // store completion + signal
  tt[3] += 1;
}

__device__ __forceinline__ void ldg256_cg(const void* p, uint32_t (&r)[8]) {   // L2 only: the slabs are rewritten by other SMs
  asm volatile("ld.global.cg.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "l"(p)
               : "memory");
}
__device__ __forceinline__ void stg256(void* p, const uint32_t (&r)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]),
               "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}

// In-place tile (two 16-bit input streams, two output streams, 256 columns) without TMA: thread = accumulator row, a warp owns
// 64 columns = four 16-column steps of one 32-byte vector per stream; the loads of step k + 2 are in flight while step k is
// computed.  in0 / in1 / out0 / out1 point at this thread's row (element offset of the warp's first column included) or are
// nullptr for rows beyond T.  Ends with every lane's stores fenced and ONE release by lane 0.
template <class Epi>
__device__ __forceinline__ void mega_inplace_direct(const Epi& epi, uint32_t taddr, uint64_t* tmem_full, uint32_t full_phase,
                                                    uint32_t tmem_empty_remote, int lane, int col0, const uint16_t* in0,
                                                    const uint16_t* in1, uint16_t* out0, uint16_t* out1, MegaSig sig,
                                                    uint32_t* tt) {
  uint32_t buf[2][2][8];   // [step parity][stream][8]
  const bool valid = out0 != nullptr;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    if (Epi::kIn > 0 && valid) {
      ldg256_cg(in0 + 16 * k, buf[k][0]);
      ldg256_cg(in1 + 16 * k, buf[k][1]);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) buf[k][0][j] = buf[k][1][j] = 0u;
    }
  }
  const uint32_t c_a = (uint32_t)clock();
  mbar_wait(tmem_full, full_phase);
  tc_fence_after();
  const uint32_t c_b = (uint32_t)clock();
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    float v[16];
    tmem_ld16(taddr + 16 * k, v);
    if (k == 3) {
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tmem_empty_remote);
    }
    uint32_t o[2][8];
    if constexpr (Epi::kIn > 0) epi.compute(col0 + 16 * k, v, buf[k & 1], o);
    else epi.compute(col0 + 16 * k, v, o);
    if (Epi::kIn > 0 && k + 2 < 4 && valid) {
      ldg256_cg(in0 + 16 * (k + 2), buf[k & 1][0]);
      ldg256_cg(in1 + 16 * (k + 2), buf[k & 1][1]);
    }
    if (valid) {
      stg256(out0 + 16 * k, o[0]);
      stg256(out1 + 16 * k, o[1]);
    }
  }
  const uint32_t c_c = (uint32_t)clock();
  __threadfence();          // this lane's stores are visible device-wide ...
  __syncwarp();             // ... before lane 0 publishes the tile
  if (lane == 0) mega_signal(sig);
  __syncwarp();
  tt[0] += c_b - c_a;
  tt[1] += c_c - c_b;
  tt[2] += (uint32_t)clock() - c_c;
  tt[3] += 1;
}

// Residual tile on a single 16-bit stream (AddTcEpi).  The caller has issued BOTH 32-column chunks of the layer input into the
// warp's two staging buffers (one mbarrier phase); each chunk is updated in place and stored.
__device__ __forceinline__ void mega_res1_task(const AddTcEpi& epi, uint32_t tmem_tile, uint64_t* tmem_full, uint32_t full_phase,
                                               uint32_t tmem_empty_remote, int q, int cg, int lane, uint32_t wbuf, uint64_t* ibar,
                                               uint32_t& it, const CUtensorMap* om, int b, int r0, MegaSig sig, uint32_t* tt,
                                               bool dead = false) {
  const uint32_t taddr = tmem_tile + ((uint32_t)(q * 32) << 16) + cg * (MEGA_BN / 4);
  const uint32_t c_a = (uint32_t)clock();
  mbar_wait(tmem_full, full_phase);
  tc_fence_after();
  mbar_wait(ibar, it & 1);
  ++it;
  const uint32_t c_b = (uint32_t)clock();
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int c0 = cg * (MEGA_BN / 4) + 32 * k;
    const uint32_t buf = wbuf + k * TC_CHUNK16_BYTES;
    uint32_t in[16];
    stage_load16(buf, lane, in);
    __syncwarp();
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float v[16];
      tmem_ld16(taddr + 32 * k + 16 * h, v);
      if (h == 1 && k == 1) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(tmem_empty_remote);
      }
      uint32_t inh[1][8], o[1][8];
#pragma unroll
      for (int j = 0; j < 8; ++j) inh[0][j] = in[8 * h + j];
      epi.compute(c0 + 16 * h, v, inh, o);
      if (dead) {
#pragma unroll
        for (int j = 0; j < 8; ++j) o[0][j] = 0u;
      }
      stage_store16h(buf, lane, h, o[0]);
    }
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) {
      tma_store_4d(om, buf, c0, r0, 0, b);
      bulk_commit();
    }
  }
  const uint32_t c_c = (uint32_t)clock();
  if (lane == 0) {
    bulk_wait_all();            // stores COMPLETE: the results are in global memory
    mega_signal(sig);
  }
  __syncwarp();
  tt[0] += c_b - c_a;
  tt[1] += c_c - c_b;
  tt[2] += (uint32_t)clock() - c_c;
  tt[3] += 1;
}

constexpr int MEGA_END_MAXC = 16;   // output channels of the fused `end` conv (2 * in_channels; every shipped config has <= 8)

// Skip tile with the `end` 1x1 conv in its epilogue.  A warp owns 32 rows x 64 of the tile's 256 skip channels: it folds its
// columns into NC partial outputs per row (weights are warp-uniform loads, L1 resident), the four warps of a TMEM lane quadrant
// meet through their staging buffers and a 128-thread named barrier, and the first of them writes the (B, cout, T) rows --
// 32 consecutive time steps per output channel, one coalesced 128-byte store each.
template <int NC>
__device__ __noinline__ void mega_end_task(const MegaParams& p, uint32_t tmem_tile, uint64_t* tmem_full, uint32_t full_phase,
                                              uint32_t tmem_empty_remote, int q, int cg, int lane, uint8_t* epi_base, int WB,
                                              int b, int r0) {
  const uint32_t taddr = tmem_tile + ((uint32_t)(q * 32) << 16) + cg * (MEGA_BN / 4);
  const int e = cg * 4 + q;
  const uint32_t wbuf = smem_u32(epi_base + e * WB);
  float acc[NC];
#pragma unroll
  for (int o = 0; o < NC; ++o) acc[o] = 0.f;
  mbar_wait(tmem_full, full_phase);
  tc_fence_after();
#pragma unroll 1
  for (int k = 0; k < 2; ++k) {
    const int c0 = cg * (MEGA_BN / 4) + 32 * k;
    if (p.store_skip && k > 0) {
      if (lane == 0) bulk_wait_read<0>();
      __syncwarp();
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float v[16];
      tmem_ld16(taddr + 32 * k + 16 * h, v);
      if (h == 1 && k == 1) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(tmem_empty_remote);
      }
      const float* w = p.w_end + c0 + 16 * h;
#pragma unroll
      for (int o = 0; o < NC; ++o) {
        float a = acc[o];
#pragma unroll
        for (int j = 0; j < 16; ++j) a = fmaf(v[j], __ldg(w + o * MEGA_BN + j), a);
        acc[o] = a;
      }
      if (p.store_skip) {
        uint32_t ov[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) ov[j] = __float_as_uint(v[j]);
        stage_store32h(wbuf, lane, h, ov);
      }
    }
    if (p.store_skip) {
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        tma_store_4d(&p.skip_c32, wbuf, c0, r0, 0, b);
        bulk_commit();
      }
    }
  }
  if (p.store_skip) {   // the staging doubles as the exchange buffer: the last store must have read it
    if (lane == 0) bulk_wait_read<0>();
    __syncwarp();
  }
  float* part = reinterpret_cast<float*>(epi_base + e * WB);
#pragma unroll
  for (int o = 0; o < NC; ++o) part[o * 32 + lane] = acc[o];
  asm volatile("bar.sync %0, 128;" ::"r"(1 + q) : "memory");
  if (cg == 0) {
    const int t = r0 + lane;
#pragma unroll
    for (int o = 0; o < NC; ++o) {
      float sacc = 0.f;
#pragma unroll
      for (int g = 0; g < 4; ++g) sacc += reinterpret_cast<const float*>(epi_base + (g * 4 + q) * WB)[o * 32 + lane];
      if (o < p.cout && t < p.T) p.lst[((long long)b * p.cout + o) * p.T + t] = sacc;
    }
  }
  asm volatile("bar.sync %0, 128;" ::"r"(1 + q) : "memory");   // the partials have been read: staging may be reused
}

template <bool SAVE>
constexpr int mega_warp_bytes() { return 2 * TC_CHUNK16_BYTES; }
constexpr int MEGA_STAGE_BYTES = TC_A_BYTES + (MEGA_BN / 2) * 128;
template <bool SAVE>
constexpr int mega_stages() {
  return (TC_SMEM_LIMIT - 1024 - TC_BAR_BYTES - TC_EPI_WARPS * mega_warp_bytes<SAVE>()) / MEGA_STAGE_BYTES;
}
template <bool SAVE>
constexpr size_t mega_smem_bytes() {
  return (size_t)mega_stages<SAVE>() * MEGA_STAGE_BYTES + TC_EPI_WARPS * mega_warp_bytes<SAVE>() + TC_BAR_BYTES + 1024;
}

// VARLEN: per-item lengths (rt_tab / row_len set); a separate instance, so the dense kernel carries none of it
template <bool SAVE, bool VARLEN = false>
__global__ void __launch_bounds__(MEGA_THREADS, 1) wn_fwd_mega_kernel(const __grid_constant__ MegaParams p) {
  extern __shared__ uint8_t smem_raw[];
  constexpr int STAGES = mega_stages<SAVE>();
  constexpr int WB = mega_warp_bytes<SAVE>();
  static_assert(STAGES >= 3, "staging leaves no room for the operand pipeline");
  static_assert(2 * TC_CHUNK16_BYTES >= TC_CHUNK32_BYTES, "fp32 chunk must fit the per-warp staging");
  const TcSmem s = tc_carve<STAGES>(smem_raw, MEGA_STAGE_BYTES, TC_EPI_WARPS * WB);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  uint32_t* done_cnt = s.tmem_ptr + 2;  // [4] per-task arrival counters of the epilogue warps (barrier area)
  static_assert((2 * STAGES + 4 + TC_EPI_WARPS) * 8 + 8 + 4 * 4 + 8 <= TC_BAR_BYTES, "barrier area too small");
  uint32_t* cleared = s.tmem_ptr + 6;   // tasks whose dependencies the scout has seen satisfied
  if (threadIdx.x < 4) done_cnt[threadIdx.x] = 0;
  if (threadIdx.x == 4) *cleared = 0;
  pdl_trigger();
  tc_setup<STAGES>(s, warp, lane, 2 * MEGA_BN, TC_EPI_WARPS);
  const uint32_t tmem_base = *s.tmem_ptr;
  pdl_wait();
  const int Crp = p.kb_h * TC_BK;
  const uint32_t gtarget = (uint32_t)p.ngt * 2u * TC_EPI_WARPS, rtarget = 2u * TC_EPI_WARPS;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      long long w_slot = 0, w_flag = 0;
      uint32_t ntask = 0;
      const long long c_start = clock64();
      const uint32_t full0 = mapa_shared(smem_u32(&s.full[0]), 0);
      const bool both = p.dual == 0;
      auto load = [&](const CUtensorMap* am, int ak, int at, int ab, const CUtensorMap* bm, int bk, int bn) {
        if (p.clk) {
          const long long c0 = clock64();
          mbar_wait(&s.empty[stage], phase ^ 1);
          w_slot += clock64() - c0;
        } else {
          mbar_wait(&s.empty[stage], phase ^ 1);
        }
        const uint32_t sa = smem_u32(s.stages + stage * MEGA_STAGE_BYTES);
        if (rank == 0) mbar_arrive_expect_tx(&s.full[stage], 2 * MEGA_STAGE_BYTES);
        const uint32_t bar = full0 + 8 * stage;
        tma_load_4d(sa, am, bar, ak, at, 0, ab);
        if (both) tma_load_2d(sa + TC_A_BYTES, bm, bar, bk, bn);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      };
      for (int task = pair; task < p.total_tasks; task += npairs) {
        const MegaTask t = mega_decode(p, task);
        if (t.type == MEGA_NONE) continue;
        const MegaTile mt = mega_tile(VARLEN ? p.rt_tab : nullptr, p.tiles_per_batch, t.rt);
        const int b = mt.b, tb = mt.tb;
        const int t0 = tb * (2 * TC_BM) + rank * TC_BM;
        const int nrow = rank * (MEGA_BN / 2);
        const long long cf = clock64();
        if (p.dual) {
          mega_wait_cleared(cleared, ++ntask);       // the scout (warp MEGA_SWARP) has done the waiting
        } else if (t.type == MEGA_G) {
          if (t.layer > 0 && !(p.dbg & 1)) {
            const uint32_t* f1 = mega_rflag(p, t.layer - 1, t.rt);
            mega_wait_flags3(tb > 0 ? f1 - 1 : f1, f1, tb + 1 < mt.ntb ? f1 + 1 : f1, rtarget, !(p.dbg & 32));
            if (!(p.dbg & 16)) fence_proxy_async_all();
          }
        } else {
          if (!(p.dbg & 1)) mega_wait_flag(mega_gflag(p, t.type == MEGA_R ? t.layer : p.depth - 1, t.rt), gtarget);
          if (!(p.dbg & 16)) fence_proxy_async_all();
        }
        w_flag += clock64() - cf;
        const bool f0 = p.fold0 && t.layer == 0;
        if (t.type == MEGA_G) {
          const int n0 = t.nt * MEGA_BN + nrow;
          if (f0) {
            for (int kb = 0; kb < p.kb_c; ++kb) load(&p.cond_op, kb * TC_BK, t0, b, &p.pa0f, kb * TC_BK, n0);
          } else {
            for (int sg = 0; sg < p.taps; ++sg) {
              const int shift = (sg - (p.taps - 1) / 2) * (1 << t.layer);
              for (int kb = 0; kb < p.kb_h; ++kb)
                load(&p.hin_op[t.layer], kb * TC_BK, t0 + shift, b, &p.pa[t.layer], sg * Crp + kb * TC_BK, n0);
            }
            for (int kb = 0; kb < p.kb_c; ++kb)
              load(&p.cond_op, kb * TC_BK, t0, b, &p.pa[t.layer], p.taps * Crp + kb * TC_BK, n0);
          }
        } else if (t.type == MEGA_R) {
          const CUtensorMap* bm = f0 ? &p.pb0f : &p.pb[t.layer];
          for (int kb = 0; kb < p.kb_g; ++kb) load(&p.g_op[t.layer], kb * TC_BK, t0, b, bm, kb * TC_BK, nrow);
          if (f0) load(&p.cond_op, (p.kb_c - 1) * TC_BK, t0, b, bm, p.kb_g * TC_BK, nrow);
        } else {
          for (int j = 0; j < p.depth; ++j)
            for (int kb = 0; kb < p.kb_g; ++kb)
              load(&p.g_op[j], kb * TC_BK, t0, b, &p.ps, (j * p.kb_g + kb) * TC_BK, nrow);
        }
      }
      if (p.clk) {
        long long* o = p.clk + ((size_t)blockIdx.x * 18 + warp) * 16;
        o[0] = w_slot; o[1] = w_flag; o[12] = clock64() - c_start;
      }
    }
  } else if (warp == MEGA_SWARP) {
    if (lane == 0 && p.dual) {
      uint32_t n = 0;
      for (int task = pair; task < p.total_tasks; task += npairs) {
        const MegaTask t = mega_decode(p, task);
        if (t.type == MEGA_NONE) continue;
        if (t.type == MEGA_G) {
          if (t.layer > 0) {
            const MegaTile mt = mega_tile(VARLEN ? p.rt_tab : nullptr, p.tiles_per_batch, t.rt);
            const uint32_t* f1 = mega_rflag(p, t.layer - 1, t.rt);
            mega_wait_flags3(mt.tb > 0 ? f1 - 1 : f1, f1, mt.tb + 1 < mt.ntb ? f1 + 1 : f1, rtarget);
          }
        } else {
          mega_wait_flag(mega_gflag(p, t.type == MEGA_R ? t.layer : p.depth - 1, t.rt), gtarget);
        }
        st_release_cta_u32(cleared, ++n);
      }
    }
  } else if (warp == MEGA_BWARP) {
    if (lane == 0 && p.dual) {
      // weight tiles of the same task sequence: no dependencies, only free ring slots
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t full0 = mapa_shared(smem_u32(&s.full[0]), 0);
      auto loadb = [&](const CUtensorMap* bm, int bk, int bn) {
        mbar_wait(&s.empty[stage], phase ^ 1);
        tma_load_2d(smem_u32(s.stages + stage * MEGA_STAGE_BYTES) + TC_A_BYTES, bm, full0 + 8 * stage, bk, bn);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      };
      for (int task = pair; task < p.total_tasks; task += npairs) {
        const MegaTask t = mega_decode(p, task);
        if (t.type == MEGA_NONE) continue;
        const int nrow = rank * (MEGA_BN / 2);
        const bool f0 = p.fold0 && t.layer == 0;
        if (t.type == MEGA_G) {
          const int n0 = t.nt * MEGA_BN + nrow;
          const int nkb = f0 ? p.kb_c : p.taps * p.kb_h + p.kb_c;
          const CUtensorMap* bm = f0 ? &p.pa0f : &p.pa[t.layer];
          for (int kb = 0; kb < nkb; ++kb) loadb(bm, kb * TC_BK, n0);
        } else if (t.type == MEGA_R) {
          const CUtensorMap* bm = f0 ? &p.pb0f : &p.pb[t.layer];
          for (int kb = 0; kb < p.kb_g + (f0 ? 1 : 0); ++kb) loadb(bm, kb * TC_BK, nrow);
        } else {
          for (int kb = 0; kb < p.depth * p.kb_g; ++kb) loadb(&p.ps, kb * TC_BK, nrow);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      long long w_empty = 0, w_full = 0;
      const long long c_start = clock64();
      for (int task = pair; task < p.total_tasks; task += npairs) {
        const MegaTask t = mega_decode(p, task);
        if (t.type == MEGA_NONE) continue;
        const bool f0 = p.fold0 && t.layer == 0;
        const int total_kb = t.type == MEGA_G ? (f0 ? p.kb_c : p.taps * p.kb_h + p.kb_c)
                                              : (t.type == MEGA_R ? p.kb_g + (f0 ? 1 : 0) : p.depth * p.kb_g);
        long long c0 = clock64();
        mbar_wait(&s.tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        w_empty += clock64() - c0;
        const uint32_t d_tmem = tmem_base + acc * MEGA_BN;
        // the conditioning's channels are padded to whole k-blocks with zeros (80 -> 128): the K = 16 steps that would
        // multiply nothing but padding are not issued (3 of the 56 steps of a gate tile at the LJ config)
        const int kb_trim = (t.type == MEGA_G || (t.type == MEGA_R && f0)) ? total_kb - 1 : -1;
        const int nk_trim = f0 ? p.kc_last0 : p.kc_last;
        for (int kb = 0; kb < total_kb; ++kb) {
          c0 = clock64();
          mbar_wait(&s.full[stage], phase);
          tc_fence_after();
          w_full += clock64() - c0;
          const uint32_t sa = smem_u32(s.stages + stage * MEGA_STAGE_BYTES);
          const uint64_t adesc = make_smem_desc(sa, p.desc_lbo, p.desc_sbo);
          const uint64_t bdesc = make_smem_desc(sa + TC_A_BYTES, p.desc_lbo, p.desc_sbo);
          const int nk = kb == kb_trim ? nk_trim : TC_BK / 16;
#pragma unroll
          for (int k = 0; k < TC_BK / 16; ++k)
            if (k < nk) umma_f16(d_tmem, adesc + 2 * k, bdesc + 2 * k, p.idesc, (kb > 0 || k > 0) ? 1u : 0u);
          umma_commit(&s.empty[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&s.tmem_full[acc]);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
      if (p.clk) {
        long long* o = p.clk + ((size_t)blockIdx.x * 18 + warp) * 16;
        o[0] = w_empty; o[1] = w_full; o[12] = clock64() - c_start;
      }
    }
  } else {
    const int e = warp - 2;
    const int q = warp & 3;
    const int cg = e >> 2;
    const uint32_t wbuf = smem_u32(s.epi + e * WB);
    uint64_t* ibar = s.in_bar + e;
    const uint32_t tmem_empty_addr = mapa_shared(smem_u32(&s.tmem_empty[0]), 0);
    const GateTcEpi<SAVE> gate_epi{nullptr, p.Cd, p.f16, p.gate_mix};
    const SplitTcEpi<true> split_epi{nullptr, p.f16};
    const AddTcEpi add_epi{nullptr, p.f16};
    const RoundTcEpi round_epi{p.f16};
    const StoreTcEpi store_epi{nullptr, nullptr};
    int acc = 0;
    uint32_t acc_phase = 0;
    uint32_t it = 0;
    uint32_t seq = 0;  // units done by this pair; warps of a CTA are never more than two units apart (TMEM double buffer)
    uint32_t tt[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};   // 32-bit cycle counters: a launch is far below 2^32 cycles
    const uint32_t c_start = (uint32_t)clock();
    MegaSig pending{nullptr, 0};
    MegaSig* prev = p.lagged ? &pending : nullptr;
    bool prev_alt = false;  // the previous unit staged through ONE of the two 2 KB buffers (gate tile without saves)
    for (int task = pair; task < p.total_tasks; task += npairs) {
      const MegaTask t = mega_decode(p, task);
      if (t.type == MEGA_NONE) continue;
      const MegaTile mt = mega_tile(VARLEN ? p.rt_tab : nullptr, p.tiles_per_batch, t.rt);
      const int b = mt.b, tb = mt.tb;
      const int r0 = tb * (2 * TC_BM) + rank * TC_BM + q * 32;
      const bool dead = VARLEN && mega_dead_row(p.row_len, b, r0 + lane);
      const uint32_t tile = tmem_base + acc * MEGA_BN;
      const uint32_t te = tmem_empty_addr + 8 * acc;
      const uint32_t dcnt = smem_u32(done_cnt + (seq & 3));
      const bool alt = !SAVE && t.type == MEGA_G;
      const uint32_t ubuf = wbuf + (alt ? (seq & 1) * TC_CHUNK16_BYTES : 0);
      ++seq;
      if (p.dbg & 8) {  // timing experiment: no epilogue work at all
        mbar_wait(&s.tmem_full[acc], acc_phase);
        tc_fence_after();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(te);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
        continue;
      }
      // lagged mode: the previous unit's stores may still be reading its staging (not if both use alternate buffers)
      if (p.lagged && !(alt && prev_alt)) {
        if (lane == 0) bulk_wait_read<0>();
        __syncwarp();
      }
      prev_alt = alt;
      if (t.type == MEGA_G) {
        mega_epilogue_task<GateTcEpi<SAVE>, MEGA_BN / 2>(gate_epi, tile, &s.tmem_full[acc], acc_phase, te, q, cg, lane, ubuf,
                                                         ibar, it, &p.g_c16[t.layer], &p.b_c16[t.layer], nullptr,
                                                         nullptr, nullptr, b, r0, t.nt * (MEGA_BN / 2),
                                                         MegaSig{mega_gflag(p, t.layer, t.rt), dcnt}, prev, p.dbg, tt);
      } else if (t.type == MEGA_R && p.res_direct && p.res_lo) {
        if (lane == 0 && !(p.dbg & 1)) mega_wait_flag(mega_gflag(p, t.layer, t.rt), gtarget);  // implies R(layer-1, rt) is complete
        __syncwarp();
        const int trow = r0 + lane;                      // row within the batch item
        const bool ok = trow < p.T;
        const size_t off = ((size_t)b * p.T + trow) * MEGA_BN + cg * (MEGA_BN / 4);
        mega_inplace_direct<SplitTcEpi<true>>(split_epi, tile + ((uint32_t)(q * 32) << 16) + cg * (MEGA_BN / 4), &s.tmem_full[acc],
                                              acc_phase, te, lane, cg * (MEGA_BN / 4), ok ? p.hi_ptr[t.layer] + off : nullptr,
                                              ok ? p.lo_ptr[t.layer] + off : nullptr,
                                              ok ? p.hi_out_ptr[t.layer + 1] + off : nullptr,
                                              ok ? p.lo_ptr[t.layer + 1] + off : nullptr,
                                              MegaSig{mega_rflag(p, t.layer, t.rt), dcnt}, tt + 4);
      } else if (t.type == MEGA_R && p.fold0 && t.layer == 0) {
        // h_1 = W_res g_0 + W_start x_a, all of it from the tensor core: nothing to load, one 16-bit stream to store
        mega_epilogue_task<RoundTcEpi, MEGA_BN>(round_epi, tile, &s.tmem_full[acc], acc_phase, te, q, cg, lane, wbuf, ibar, it,
                                                &p.hi_c16[1], nullptr, nullptr, nullptr, nullptr, b, r0, 0,
                                                MegaSig{mega_rflag(p, 0, t.rt), dcnt}, prev, p.dbg, tt + 4, dead);
      } else if (t.type == MEGA_R && !p.res_lo) {
        if (lane == 0) {  // the warp's whole share of the layer input (two chunks), ahead of the accumulator
          mega_wait_flag(mega_gflag(p, t.layer, t.rt), gtarget);  // implies R(layer-1, rt) is complete
          fence_proxy_async_all();
          mbar_arrive_expect_tx(ibar, 2 * TC_CHUNK16_BYTES);
          const int c0 = cg * (MEGA_BN / 4);
          tma_load_4d_local(wbuf, &p.hi_c16[t.layer], smem_u32(ibar), c0, r0, 0, b);
          tma_load_4d_local(wbuf + TC_CHUNK16_BYTES, &p.hi_c16[t.layer], smem_u32(ibar), c0 + 32, r0, 0, b);
        }
        __syncwarp();
        mega_res1_task(add_epi, tile, &s.tmem_full[acc], acc_phase, te, q, cg, lane, wbuf, ibar, it, &p.hi_c16[t.layer + 1], b, r0,
                       MegaSig{mega_rflag(p, t.layer, t.rt), dcnt}, tt + 4, dead);
      } else if (t.type == MEGA_R) {
        if (lane == 0) {  // chunk 0 of the layer input's (hi, lo) pair, ahead of the accumulator
          if (!(p.dbg & 1)) mega_wait_flag(mega_gflag(p, t.layer, t.rt), gtarget);  // implies R(layer-1, rt) is complete
          fence_proxy_async_all();
          mbar_arrive_expect_tx(ibar, 2 * TC_CHUNK16_BYTES);
          const int c0 = cg * (MEGA_BN / 4);
          tma_load_4d_local(ubuf, &p.hi_c16[t.layer], smem_u32(ibar), c0, r0, 0, b);
          tma_load_4d_local(ubuf + TC_CHUNK16_BYTES, &p.lo_c16[t.layer], smem_u32(ibar), c0, r0, 0, b);
        }
        __syncwarp();
        mega_epilogue_task<SplitTcEpi<true>, MEGA_BN>(split_epi, tile, &s.tmem_full[acc], acc_phase, te, q, cg, lane, ubuf, ibar,
                                                      it, &p.hi_c16[t.layer + 1], &p.lo_c16[t.layer + 1], nullptr,
                                                      &p.hi_c16[t.layer], &p.lo_c16[t.layer], b, r0, 0,
                                                      MegaSig{mega_rflag(p, t.layer, t.rt), dcnt}, prev, p.dbg, tt + 4, dead);
      } else if (p.lst != nullptr) {
        if (p.lagged) {   // staging is about to be used as plain memory: no store may still be reading it
          if (lane == 0) bulk_wait_read<0>();
          __syncwarp();
        }
        if (p.cout <= 8) mega_end_task<8>(p, tile, &s.tmem_full[acc], acc_phase, te, q, cg, lane, s.epi, WB, b, r0);
        else mega_end_task<MEGA_END_MAXC>(p, tile, &s.tmem_full[acc], acc_phase, te, q, cg, lane, s.epi, WB, b, r0);
      } else {
        mega_epilogue_task<StoreTcEpi, MEGA_BN>(store_epi, tile, &s.tmem_full[acc], acc_phase, te, q, cg, lane, ubuf, ibar, it,
                                                &p.skip_c32, nullptr, nullptr, nullptr, nullptr, b, r0, 0,
                                                MegaSig{nullptr, dcnt}, prev, p.dbg, tt + 8);
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (lane == 0) {  // flush: the last unit's stores, and its signal in lagged mode
      bulk_wait_all();
      if (p.lagged) mega_signal(pending);
      if (p.clk) {
        long long* o = p.clk + ((size_t)blockIdx.x * 18 + warp) * 16;
        for (int i = 0; i < 12; ++i) o[i] = tt[i];
        o[12] = (uint32_t)clock() - c_start;
      }
    }
  }
  tc_teardown(tmem_base, warp, 2 * MEGA_BN);
}


// ================================================================================================
// Backward chain of the WN as one task kernel (same machinery, the reversible backward's dgrad path):
//     DG(i, rt)  dgate GEMM  dg = [dh_{i+1} | dskip] W_o,  epilogue dpre = dg * d(tanh * sigmoid) from the saved values
//     DX(i, rt)  dx GEMM     dh_i = dh_{i+1} + sum_tap dpre_i[row - shift] W_tap   (epilogue adds the (hi, lo) pair)
// for layers depth-1 .. 0.  DG(i, rt) needs DX(i+1, rt); DX(i, rt) needs DG(i, rt-1 .. rt+1).  List: the RT tiles
// DG(depth-1, *) (they depend on nothing but dskip), then slots u = j * RT + rt (layer i = depth-1-j) holding
// [DX(u), DG of the layer below for tile u - lag]; pair p takes entry k * P + ((p - k) mod P) in round k (the skew
// keeps a pair from seeing only one kind of entry: P is even and so is the slot size).  The weight-gradient GEMMs
// and the conditioning-gradient GEMM run afterwards from the per-layer dpre / dh slabs this kernel leaves behind.
// ================================================================================================
enum { MEGA_DG = 0, MEGA_DX = 1 };

struct alignas(64) MegaBwdParams {
  CUtensorMap dh_op[MEGA_D];      // operand maps: dh_i hi halves (dh_op[i] feeds DG(i-1))
  CUtensorMap dskip_op;           // operand map: gradient of the cumulative skip
  CUtensorMap dpre_op[MEGA_D];    // operand maps: dpre_i [rows][2Cd]
  CUtensorMap q1[MEGA_D], q2[MEGA_D];                       // W_o^T and W^T (per tap) weights
  CUtensorMap sa_c16[MEGA_D], sb_c16[MEGA_D];               // chunk maps: gate output g / saved sigmoid (GateBwdTcEpi)
  CUtensorMap dpt_c16[MEGA_D], dps_c16[MEGA_D];             // chunk maps: tanh / sigmoid halves of dpre_i
  CUtensorMap dhi_c16[MEGA_D], dlo_c16[MEGA_D];             // chunk maps: (hi, lo) pair of dh_i
  uint32_t* flags;                // [depth][2][RT]: DG-done / DX-done counters (zeroed before the launch)
  int depth, B, T, tiles_per_batch, RT;
  int taps, kb_r, kb_s, kb_d2;    // taps; k-blocks of dh / dskip / dpre (2Cd)
  int f16;
  uint32_t idesc, desc_lbo, desc_sbo;
  int lag, total_tasks;
  int dual;                       // see MegaParams::dual
  // direct global loads / stores in the epilogues (see MegaParams::res_direct)
  const uint16_t* sa_ptr[MEGA_D];   // gate output g  [rows][Cd]
  const uint16_t* sb_ptr[MEGA_D];   // saved sigmoid  [rows][Cd]
  uint16_t* dpre_ptr[MEGA_D];       // dpre_i         [rows][2Cd]
  uint16_t* dhi_ptr[MEGA_D];        // dh_i hi halves [rows][Cr]
  uint16_t* dlo_ptr[MEGA_D];        // dh_i lo halves [rows][Cr]
  int direct;
  int res_lo;                       // see MegaParams::res_lo (here: the residual GRADIENT stream)
  // `end` conv folded into the dgate GEMM (PackedLayout::Q1f): instead of the kb_s k-blocks of dskip = W_end^T d(log_s, t), a
  // dgate tile reads ONE k-block of the slab dl = S * d(log_s, t) (2 in_channels real columns) against (W_end W_skip)^T
  int fold_end;
  int kdl;                          // K = 16 steps of that k-block that hold real columns
  CUtensorMap dl_op;
  CUtensorMap q1f[MEGA_D];
};

__host__ __device__ __forceinline__ MegaTask mega_bwd_decode(const MegaBwdParams& p, int idx) {
  MegaTask t;
  t.nt = 0;
  if (idx < p.RT) {
    t.type = MEGA_DG; t.layer = p.depth - 1; t.rt = idx;
    return t;
  }
  idx -= p.RT;
  const int sl = idx >> 1, w = idx & 1;
  const int u = w == 0 ? sl : sl - p.lag;
  const int j = u >= 0 ? u / p.RT : 0;
  t.rt = u - j * p.RT;
  t.layer = p.depth - 1 - j;
  if (w == 0) {
    t.type = u < p.depth * p.RT ? MEGA_DX : MEGA_NONE;
  } else {
    t.type = (u >= 0 && t.layer >= 1 && j < p.depth) ? MEGA_DG : MEGA_NONE;
    t.layer -= 1;  // the dgate GEMM of the layer below
  }
  return t;
}
__device__ __forceinline__ int mega_bwd_entry(int total, int k, int pair, int npairs) {
  int r = (pair - k) % npairs;
  if (r < 0) r += npairs;
  const int e = k * npairs + r;
  return e < total ? e : -1;
}
__device__ __forceinline__ uint32_t* mega_bwd_gflag(const MegaBwdParams& p, int layer, int rt) {
  return p.flags + (size_t)(2 * layer) * p.RT + rt;
}
__device__ __forceinline__ uint32_t* mega_bwd_xflag(const MegaBwdParams& p, int layer, int rt) {
  return p.flags + (size_t)(2 * layer + 1) * p.RT + rt;
}

constexpr int MEGA_BWD_WARP_BYTES = 2 * TC_CHUNK16_BYTES;
constexpr int MEGA_BWD_STAGES = (TC_SMEM_LIMIT - 1024 - TC_BAR_BYTES - TC_EPI_WARPS * MEGA_BWD_WARP_BYTES) / MEGA_STAGE_BYTES;
constexpr size_t MEGA_BWD_SMEM_BYTES =
    (size_t)MEGA_BWD_STAGES * MEGA_STAGE_BYTES + TC_EPI_WARPS * MEGA_BWD_WARP_BYTES + TC_BAR_BYTES + 1024;

__global__ void __launch_bounds__(MEGA_THREADS, 1) wn_bwd_mega_kernel(const __grid_constant__ MegaBwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  constexpr int STAGES = MEGA_BWD_STAGES;
  constexpr int WB = MEGA_BWD_WARP_BYTES;
  const TcSmem s = tc_carve<STAGES>(smem_raw, MEGA_STAGE_BYTES, TC_EPI_WARPS * WB);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  uint32_t* done_cnt = s.tmem_ptr + 2;
  static_assert((2 * STAGES + 4 + TC_EPI_WARPS) * 8 + 8 + 4 * 4 + 8 <= TC_BAR_BYTES, "barrier area too small");
  uint32_t* cleared = s.tmem_ptr + 6;
  if (threadIdx.x < 4) done_cnt[threadIdx.x] = 0;
  if (threadIdx.x == 4) *cleared = 0;
  pdl_trigger();
  tc_setup<STAGES>(s, warp, lane, 2 * MEGA_BN, TC_EPI_WARPS);
  const uint32_t tmem_base = *s.tmem_ptr;
  pdl_wait();
  const uint32_t target = 2u * TC_EPI_WARPS;
  const int rounds = (p.total_tasks + npairs - 1) / npairs;
  const int Crp = p.kb_r * TC_BK, Cd2p = p.kb_d2 * TC_BK;

  if (warp == 0) {
    if (lane == 0) {
      uint32_t ntask = 0;
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t full0 = mapa_shared(smem_u32(&s.full[0]), 0);
      const bool both = p.dual == 0;
      auto load = [&](const CUtensorMap* am, int ak, int at, int ab, const CUtensorMap* bm, int bk, int bn) {
        mbar_wait(&s.empty[stage], phase ^ 1);
        const uint32_t sa = smem_u32(s.stages + stage * MEGA_STAGE_BYTES);
        if (rank == 0) mbar_arrive_expect_tx(&s.full[stage], 2 * MEGA_STAGE_BYTES);
        const uint32_t bar = full0 + 8 * stage;
        tma_load_4d(sa, am, bar, ak, at, 0, ab);
        if (both) tma_load_2d(sa + TC_A_BYTES, bm, bar, bk, bn);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      };
      for (int k = 0; k < rounds; ++k) {
        const int task = mega_bwd_entry(p.total_tasks, k, pair, npairs);
        if (task < 0) continue;
        const MegaTask t = mega_bwd_decode(p, task);
        if (t.type == MEGA_NONE) continue;
        const int b = t.rt / p.tiles_per_batch, tb = t.rt - b * p.tiles_per_batch;
        const int t0 = tb * (2 * TC_BM) + rank * TC_BM;
        const int nrow = rank * (MEGA_BN / 2);
        const bool last = t.layer == p.depth - 1;
        if (p.dual) {
          mega_wait_cleared(cleared, ++ntask);
        } else if (t.type == MEGA_DG) {
          if (!last) {
            mega_wait_flag(mega_bwd_xflag(p, t.layer + 1, t.rt), target);
            fence_proxy_async_all();
          }
        } else {
          const uint32_t* f1 = mega_bwd_gflag(p, t.layer, t.rt);
          mega_wait_flags3(tb > 0 ? f1 - 1 : f1, f1, tb + 1 < p.tiles_per_batch ? f1 + 1 : f1, target);
          fence_proxy_async_all();
        }
        if (t.type == MEGA_DG) {
          const CUtensorMap* bm = p.fold_end ? &p.q1f[t.layer] : &p.q1[t.layer];
          if (!last)
            for (int kb = 0; kb < p.kb_r; ++kb) load(&p.dh_op[t.layer + 1], kb * TC_BK, t0, b, bm, kb * TC_BK, nrow);
          if (p.fold_end) {
            load(&p.dl_op, 0, t0, b, bm, last ? 0 : Crp, nrow);
          } else {
            for (int kb = 0; kb < p.kb_s; ++kb) load(&p.dskip_op, kb * TC_BK, t0, b, bm, (last ? 0 : Crp) + kb * TC_BK, nrow);
          }
        } else {
          for (int sg = 0; sg < p.taps; ++sg) {
            const int shift = -(sg - (p.taps - 1) / 2) * (1 << t.layer);
            for (int kb = 0; kb < p.kb_d2; ++kb)
              load(&p.dpre_op[t.layer], kb * TC_BK, t0 + shift, b, &p.q2[t.layer], sg * Cd2p + kb * TC_BK, nrow);
          }
        }
      }
    }
  } else if (warp == MEGA_SWARP) {
    if (lane == 0 && p.dual) {
      uint32_t n = 0;
      for (int k = 0; k < rounds; ++k) {
        const int task = mega_bwd_entry(p.total_tasks, k, pair, npairs);
        if (task < 0) continue;
        const MegaTask t = mega_bwd_decode(p, task);
        if (t.type == MEGA_NONE) continue;
        if (t.type == MEGA_DG) {
          if (t.layer != p.depth - 1) mega_wait_flag(mega_bwd_xflag(p, t.layer + 1, t.rt), target);
        } else {
          const int tb = t.rt % p.tiles_per_batch;
          const uint32_t* f1 = mega_bwd_gflag(p, t.layer, t.rt);
          mega_wait_flags3(tb > 0 ? f1 - 1 : f1, f1, tb + 1 < p.tiles_per_batch ? f1 + 1 : f1, target);
        }
        st_release_cta_u32(cleared, ++n);
      }
    }
  } else if (warp == MEGA_BWARP) {
    if (lane == 0 && p.dual) {
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t full0 = mapa_shared(smem_u32(&s.full[0]), 0);
      auto loadb = [&](const CUtensorMap* bm, int bk, int bn) {
        mbar_wait(&s.empty[stage], phase ^ 1);
        tma_load_2d(smem_u32(s.stages + stage * MEGA_STAGE_BYTES) + TC_A_BYTES, bm, full0 + 8 * stage, bk, bn);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      };
      for (int k = 0; k < rounds; ++k) {
        const int task = mega_bwd_entry(p.total_tasks, k, pair, npairs);
        if (task < 0) continue;
        const MegaTask t = mega_bwd_decode(p, task);
        if (t.type == MEGA_NONE) continue;
        const int nrow = rank * (MEGA_BN / 2);
        if (t.type == MEGA_DG) {
          const int ks = p.fold_end ? 1 : p.kb_s;
          const int nkb = (t.layer == p.depth - 1) ? ks : p.kb_r + ks;
          const CUtensorMap* bm = p.fold_end ? &p.q1f[t.layer] : &p.q1[t.layer];
          for (int kb = 0; kb < nkb; ++kb) loadb(bm, kb * TC_BK, nrow);
        } else {
          for (int kb = 0; kb < p.taps * p.kb_d2; ++kb) loadb(&p.q2[t.layer], kb * TC_BK, nrow);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int k = 0; k < rounds; ++k) {
        const int task = mega_bwd_entry(p.total_tasks, k, pair, npairs);
        if (task < 0) continue;
        const MegaTask t = mega_bwd_decode(p, task);
        if (t.type == MEGA_NONE) continue;
        const int ks = p.fold_end ? 1 : p.kb_s;
        const int total_kb = t.type == MEGA_DX ? p.taps * p.kb_d2 : (t.layer == p.depth - 1 ? ks : p.kb_r + ks);
        const int kb_trim = (t.type == MEGA_DG && p.fold_end) ? total_kb - 1 : -1;   // the dl k-block: 2 in_channels real columns
        mbar_wait(&s.tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * MEGA_BN;
        for (int kb = 0; kb < total_kb; ++kb) {
          mbar_wait(&s.full[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(s.stages + stage * MEGA_STAGE_BYTES);
          const uint64_t adesc = make_smem_desc(sa, p.desc_lbo, p.desc_sbo);
          const uint64_t bdesc = make_smem_desc(sa + TC_A_BYTES, p.desc_lbo, p.desc_sbo);
          const int nk = kb == kb_trim ? p.kdl : TC_BK / 16;
#pragma unroll
          for (int kk = 0; kk < TC_BK / 16; ++kk)
            if (kk < nk) umma_f16(d_tmem, adesc + 2 * kk, bdesc + 2 * kk, p.idesc, (kb > 0 || kk > 0) ? 1u : 0u);
          umma_commit(&s.empty[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&s.tmem_full[acc]);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else {
    const int e = warp - 2;
    const int q = warp & 3;
    const int cg = e >> 2;
    const uint32_t wbuf = smem_u32(s.epi + e * WB);
    uint64_t* ibar = s.in_bar + e;
    const uint32_t tmem_empty_addr = mapa_shared(smem_u32(&s.tmem_empty[0]), 0);
    const GateBwdTcEpi gbwd_epi{p.f16};
    const SplitTcEpi<true> add_epi{nullptr, p.f16};
    const SplitTcEpi<false> first_epi{nullptr, p.f16};
    const AddTcEpi add1_epi{nullptr, p.f16};
    const RoundTcEpi round_epi{p.f16};
    int acc = 0;
    uint32_t acc_phase = 0;
    uint32_t it = 0, seq = 0;
    uint32_t tt[4] = {0, 0, 0, 0};
    for (int k = 0; k < rounds; ++k) {
      const int task = mega_bwd_entry(p.total_tasks, k, pair, npairs);
      if (task < 0) continue;
      const MegaTask t = mega_bwd_decode(p, task);
      if (t.type == MEGA_NONE) continue;
      const int b = t.rt / p.tiles_per_batch, tb = t.rt - b * p.tiles_per_batch;
      const int r0 = tb * (2 * TC_BM) + rank * TC_BM + q * 32;
      const uint32_t tile = tmem_base + acc * MEGA_BN;
      const uint32_t te = tmem_empty_addr + 8 * acc;
      const uint32_t dcnt = smem_u32(done_cnt + (seq++ & 3));
      const bool last = t.layer == p.depth - 1;
      const int c0 = cg * (MEGA_BN / 4);
      if (p.direct && p.res_lo) {
        const int trow = r0 + lane;
        const bool ok = trow < p.T;
        const size_t row = (size_t)b * p.T + trow;
        const uint32_t ta = tile + ((uint32_t)(q * 32) << 16) + c0;
        if (t.type == MEGA_DG) {
          const size_t oi = row * MEGA_BN + c0, oo = row * (2 * MEGA_BN) + c0;
          mega_inplace_direct<GateBwdTcEpi>(gbwd_epi, ta, &s.tmem_full[acc], acc_phase, te, lane, c0,
                                            ok ? p.sa_ptr[t.layer] + oi : nullptr, ok ? p.sb_ptr[t.layer] + oi : nullptr,
                                            ok ? p.dpre_ptr[t.layer] + oo : nullptr,
                                            ok ? p.dpre_ptr[t.layer] + oo + MEGA_BN : nullptr,
                                            MegaSig{mega_bwd_gflag(p, t.layer, t.rt), dcnt}, tt);
        } else if (!last) {
          if (lane == 0) mega_wait_flag(mega_bwd_xflag(p, t.layer + 1, t.rt), target);   // the upstream (hi, lo) pair is complete
          __syncwarp();
          const size_t o = row * MEGA_BN + c0;
          mega_inplace_direct<SplitTcEpi<true>>(add_epi, ta, &s.tmem_full[acc], acc_phase, te, lane, c0,
                                                ok ? p.dhi_ptr[t.layer + 1] + o : nullptr, ok ? p.dlo_ptr[t.layer + 1] + o : nullptr,
                                                ok ? p.dhi_ptr[t.layer] + o : nullptr, ok ? p.dlo_ptr[t.layer] + o : nullptr,
                                                MegaSig{mega_bwd_xflag(p, t.layer, t.rt), dcnt}, tt);
        } else {
          const size_t o = row * MEGA_BN + c0;
          mega_inplace_direct<SplitTcEpi<false>>(first_epi, ta, &s.tmem_full[acc], acc_phase, te, lane, c0, nullptr, nullptr,
                                                 ok ? p.dhi_ptr[t.layer] + o : nullptr, ok ? p.dlo_ptr[t.layer] + o : nullptr,
                                                 MegaSig{mega_bwd_xflag(p, t.layer, t.rt), dcnt}, tt);
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
        continue;
      }
      if (t.type == MEGA_DG) {
        if (lane == 0) {  // chunk 0 of the gate output / saved sigmoid (written by the forward: always ready)
          fence_proxy_async_all();
          mbar_arrive_expect_tx(ibar, 2 * TC_CHUNK16_BYTES);
          tma_load_4d_local(wbuf, &p.sa_c16[t.layer], smem_u32(ibar), c0, r0, 0, b);
          tma_load_4d_local(wbuf + TC_CHUNK16_BYTES, &p.sb_c16[t.layer], smem_u32(ibar), c0, r0, 0, b);
        }
        __syncwarp();
        mega_epilogue_task<GateBwdTcEpi, MEGA_BN>(gbwd_epi, tile, &s.tmem_full[acc], acc_phase, te, q, cg, lane, wbuf, ibar, it,
                                                  &p.dpt_c16[t.layer], &p.dps_c16[t.layer], nullptr, &p.sa_c16[t.layer],
                                                  &p.sb_c16[t.layer], b, r0, 0,
                                                  MegaSig{mega_bwd_gflag(p, t.layer, t.rt), dcnt}, nullptr, 0, tt);
      } else if (!last && !p.res_lo) {
        if (lane == 0) {  // the warp's whole share of the upstream residual gradient (two chunks of one stream)
          mega_wait_flag(mega_bwd_xflag(p, t.layer + 1, t.rt), target);
          fence_proxy_async_all();
          mbar_arrive_expect_tx(ibar, 2 * TC_CHUNK16_BYTES);
          tma_load_4d_local(wbuf, &p.dhi_c16[t.layer + 1], smem_u32(ibar), c0, r0, 0, b);
          tma_load_4d_local(wbuf + TC_CHUNK16_BYTES, &p.dhi_c16[t.layer + 1], smem_u32(ibar), c0 + 32, r0, 0, b);
        }
        __syncwarp();
        mega_res1_task(add1_epi, tile, &s.tmem_full[acc], acc_phase, te, q, cg, lane, wbuf, ibar, it, &p.dhi_c16[t.layer], b, r0,
                       MegaSig{mega_bwd_xflag(p, t.layer, t.rt), dcnt}, tt);
      } else if (!p.res_lo) {
        mega_epilogue_task<RoundTcEpi, MEGA_BN>(round_epi, tile, &s.tmem_full[acc], acc_phase, te, q, cg, lane, wbuf, ibar, it,
                                                &p.dhi_c16[t.layer], nullptr, nullptr, nullptr, nullptr, b, r0, 0,
                                                MegaSig{mega_bwd_xflag(p, t.layer, t.rt), dcnt}, nullptr, 0, tt);
      } else if (!last) {
        if (lane == 0) {  // chunk 0 of the upstream residual gradient's (hi, lo) pair
          mega_wait_flag(mega_bwd_xflag(p, t.layer + 1, t.rt), target);
          fence_proxy_async_all();
          mbar_arrive_expect_tx(ibar, 2 * TC_CHUNK16_BYTES);
          tma_load_4d_local(wbuf, &p.dhi_c16[t.layer + 1], smem_u32(ibar), c0, r0, 0, b);
          tma_load_4d_local(wbuf + TC_CHUNK16_BYTES, &p.dlo_c16[t.layer + 1], smem_u32(ibar), c0, r0, 0, b);
        }
        __syncwarp();
        mega_epilogue_task<SplitTcEpi<true>, MEGA_BN>(add_epi, tile, &s.tmem_full[acc], acc_phase, te, q, cg, lane, wbuf, ibar, it,
                                                      &p.dhi_c16[t.layer], &p.dlo_c16[t.layer], nullptr,
                                                      &p.dhi_c16[t.layer + 1], &p.dlo_c16[t.layer + 1], b, r0, 0,
                                                      MegaSig{mega_bwd_xflag(p, t.layer, t.rt), dcnt}, nullptr, 0, tt);
      } else {
        mega_epilogue_task<SplitTcEpi<false>, MEGA_BN>(first_epi, tile, &s.tmem_full[acc], acc_phase, te, q, cg, lane, wbuf, ibar,
                                                       it, &p.dhi_c16[t.layer], &p.dlo_c16[t.layer], nullptr, nullptr, nullptr,
                                                       b, r0, 0, MegaSig{mega_bwd_xflag(p, t.layer, t.rt), dcnt}, nullptr, 0,
                                                       tt);
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (lane == 0) bulk_wait_all();
  }
  tc_teardown(tmem_base, warp, 2 * MEGA_BN);
}

}  // namespace cmwg
