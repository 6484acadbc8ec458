// nfb_tile2.cuh — machinery shared by the kernels that keep TWO tiles in flight per SM (nfb_render2.cu: v6, nfb_render3.cu: v7):
// the per-tile-pair weight program (one LOAD per ring slot), the compile-time-unrolled MMA issue code of one stream, the
// weight producer's loop body and the epilogue of one half-step of one stream.
// See the header of nfb_render2.cu for the TMEM layout (P_x operand / Q_x accumulator per stream) and the half-step order.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <type_traits>
#include <utility>

#include "nfb_layout.h"
#include "nfb_ptx.cuh"
#include "nfb_render_common.cuh"

namespace nfb {
namespace t2 {

constexpr int kNumSlots = 9;
constexpr int kSlotBytes = 16384;
constexpr int kRingBytes = kNumSlots * kSlotBytes;
#ifndef NFB_V6_CLUSTER
#define NFB_V6_CLUSTER 2
#endif
constexpr int kCluster = NFB_V6_CLUSTER;  // CTAs sharing every weight half-unit through one multicast L2 read

// Half-steps.  Step s (nfb_layout.h) has 1 or 2 halves; half h covers weight rows [h * nh0, h * nh0 + N_h).
__host__ __device__ constexpr int num_halves(int s) { return step_info(s).nh1 > 0 ? 2 : 1; }
__host__ __device__ constexpr int half_rows(int s, int h) { return h ? step_info(s).nh1 : step_info(s).nh0; }

// The per-tile program.  A LOAD fills one ring slot: one [128 rows x 64 K] half-unit (16 KB), or — for the 16-row halves
// (sigma row block of step 6, fc_rgb) — all K atoms of the half-step as 2 KB pieces, so that a slot is never spent on 2 KB.
// 54 loads per tile pair = 6 rounds of the 9-slot ring: slot index, mbarrier parity and every shared-memory / TMEM operand
// address of the MMA issue code are therefore COMPILE-TIME constants (the issue loop is fully unrolled; it was bounding the
// tensor pipe at ~100 cycles per MMA when it read a constant-memory table and built descriptors at run time).
struct Load {
  int src[4];    // byte offset of each piece in the packed weight stream (nfb_layout.h)
  int a_col[4];  // TMEM column (relative to P_x) of each piece's A operand; -1: the positional-encoding atom (A from shared memory)
  int n_atoms;   // pieces = K atoms in this slot
  int rows;      // MMA N = weight rows per piece (128 or 16)
  int first, last, group;
};
constexpr int kMaxLoads = 56, kMaxGroups = 20;
struct LoadTable { Load l[kMaxLoads]; int gfirst[kMaxGroups], gcount[kMaxGroups]; int n, n_groups, n_pieces; };
constexpr LoadTable make_loads() {
  LoadTable t{};
  int i = 0, g = 0, pieces = 0;
  for (int s = 0; s < kNumSteps; ++s) {
    const StepInfo si = step_info(s);
    for (int h = 0; h < num_halves(s); ++h, ++g) {
      const int rows = half_rows(s, h);
      t.gfirst[g] = i;
      if (rows == kTileM) {
        for (int u = 0; u < si.k_atoms; ++u, ++i, ++pieces) {
          Load& L = t.l[i];
          L.n_atoms = 1; L.rows = rows; L.group = g;
          L.src[0] = step_offset_x1(s) + unit_offset_in_step(s, u) + h * si.nh0 * 128;
          L.a_col[0] = (si.pe_first && u == 0) ? -1 : (u - si.pe_first) * 32;
          L.first = (u == 0); L.last = (u == si.k_atoms - 1);
        }
      } else {
        Load& L = t.l[i];
        L.n_atoms = si.k_atoms; L.rows = rows; L.group = g; L.first = 1; L.last = 1;
        for (int u = 0; u < si.k_atoms; ++u, ++pieces) {
          L.src[u] = step_offset_x1(s) + unit_offset_in_step(s, u) + h * si.nh0 * 128;
          L.a_col[u] = u * 32;
        }
        ++i;
      }
      t.gcount[g] = i - t.gfirst[g];
    }
  }
  t.n = i; t.n_groups = g; t.n_pieces = pieces;
  return t;
}
constexpr LoadTable kLoads = make_loads();
constexpr int kNumLoads = kLoads.n;          // 54
constexpr int kNumGroups = kLoads.n_groups;  // 17
static_assert(kNumLoads == 54 && kNumGroups == 17 && kLoads.n_pieces == 58, "program shape");
static_assert(kNumLoads % kNumSlots == 0 && (kNumLoads / kNumSlots) % 2 == 0,
              "every tile must start at ring slot 0 with the same mbarrier parity (static slot / parity in the issue code)");
static_assert(kNumLoads % 2 == 0, "the multicast issuer alternates between the two CTAs per load");
constexpr int last_pe_group() {  // the last half-step group whose first piece is the PE atom (step 3, half 1)
  int last = -1;
  for (int i = 0; i < kLoads.n; ++i)
    if (kLoads.l[i].a_col[0] < 0) last = kLoads.l[i].group;
  return last;
}
constexpr int kLastPeGroup = last_pe_group();
static_assert(kLastPeGroup == 7, "step 3, half 1");
static __constant__ LoadTable c_loads = make_loads();  // the weight producer's copy (its loop is not unrolled)

// ---- the MMA issue code of one stream, unrolled at compile time ----------------------------------------------------
struct IssueCtx {
  uint32_t ring, p_tmem, q_tmem, bar_full, bar_empty, bar_accfull;  // ring = shared address of slot 0
  uint64_t pe_desc;
  uint32_t ring_desc_lo;  // low word of the SWIZZLE_128B descriptor of ring slot 0 (the high word is a constant)
};
// 64-bit shared-memory descriptor (K-major, SWIZZLE_128B, SBO 1024 B, version 1) from its low word
__device__ __forceinline__ uint64_t desc_from_lo(uint32_t lo) {
  uint64_t d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(0x40004040u));
  return d;
}
__device__ __forceinline__ uint32_t desc_lo_of(uint32_t smem_addr) { return ((smem_addr & 0x3FFFFu) >> 4) | (1u << 16); }
template <int I>
__device__ __forceinline__ void issue_load_mmas(const IssueCtx& c) {
  constexpr Load L = kLoads.l[I];
  constexpr int slot = I % kNumSlots;
  constexpr uint32_t idesc = umma_idesc_f16(kTileM, L.rows);
  // Launder the two bases through an empty asm: the operand addresses below are then computed next to their MMA (one add
  // each) instead of being pre-computed for the whole unrolled program and kept in (or spilled from) ~100 registers.
  uint32_t desc_lo = c.ring_desc_lo, p_tmem = c.p_tmem;
  asm volatile("" : "+r"(desc_lo), "+r"(p_tmem));
#pragma unroll
  for (int a = 0; a < L.n_atoms; ++a) {
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      // descriptor of (slot, piece a, K step ks): the start-address field (16-byte units) of slot 0's descriptor plus a
      // compile-time offset — one 32-bit add per MMA, nothing worth keeping in a register across MMAs
      const uint64_t b_desc = desc_from_lo(desc_lo + (uint32_t)((slot * kSlotBytes + a * L.rows * 128) / 16 + ks * 2));
      const uint32_t acc = (L.first && a == 0 && ks == 0) ? 0u : 1u;
      if (L.a_col[a] < 0) umma_ss(c.q_tmem, c.pe_desc + (uint64_t)(ks * 2), b_desc, idesc, acc);
      else umma_ts(c.q_tmem, p_tmem + (uint32_t)(L.a_col[a] + ks * 8), b_desc, idesc, acc);
    }
  }
  umma_commit_multicast(c.bar_empty + slot * 8, (uint16_t)((1u << kCluster) - 1));  // this stream is done with the slot
}
template <class F, int... G>
__device__ __forceinline__ void for_each_group(F& f, std::integer_sequence<int, G...>) {
  (f(std::integral_constant<int, G>{}), ...);
}
// loads [I, I + N) of one group, two loads (8 MMAs) per elected block: the whole warp waits for their weights first.
template <int I, int N>
__device__ __forceinline__ void issue_loads(const IssueCtx& c) {
  if constexpr (N > 0) {
    constexpr int K = N < 2 ? N : 2;
    mbar_wait(c.bar_full + (I % kNumSlots) * 8, (uint32_t)((I / kNumSlots) & 1));
    if constexpr (K == 2) mbar_wait(c.bar_full + ((I + 1) % kNumSlots) * 8, (uint32_t)(((I + 1) / kNumSlots) & 1));
    tc_fence_after_sync();
    if (elect_one()) {
      issue_load_mmas<I>(c);
      if constexpr (K == 2) issue_load_mmas<I + 1>(c);
      if constexpr (kLoads.l[I + K - 1].last != 0) umma_commit(c.bar_accfull);
    }
    __syncwarp();
    issue_loads<I + K, N - K>(c);
  }
}

// Accumulator chunk -> bias, ReLU, FP16: this thread's 64 columns of the half-step as 32 packed words.
__device__ __forceinline__ void epi_load64(uint32_t t_q, uint32_t bias, uint32_t extra, uint32_t (&h)[32]) {
  uint32_t va[32], vb[32], ha[16], hb[16], lo[16];
  tmem_ld32(t_q, va);
  tmem_ld32(t_q + 32, vb);
  tmem_wait_ld();
  epi_math<false>(va, bias, extra, nullptr, ha, lo);
  epi_math<false>(vb, bias + 128, extra ? extra + 128 : 0u, nullptr, hb, lo);
#pragma unroll
  for (int j = 0; j < 16; ++j) { h[j] = ha[j]; h[16 + j] = hb[j]; }
}
// Half-0 variant: the result stays in registers, so the accumulator is free as soon as it has been LOADED — the gate
// (`bar`, one arrival per warp) is signalled before the arithmetic, which then overlaps the next half-step's MMAs.
__device__ __forceinline__ void epi_load64_early(uint32_t t_q, uint32_t bias, uint32_t extra, uint32_t (&h)[32], uint32_t bar, int lane) {
  uint32_t va[32], vb[32], ha[16], hb[16], lo[16];
  tmem_ld32(t_q, va);
  tmem_ld32(t_q + 32, vb);
  tmem_wait_ld();
  tc_fence_before_sync();
  __syncwarp();
  if (lane == 0) mbar_arrive(bar);
  epi_math<false>(va, bias, extra, nullptr, ha, lo);
  epi_math<false>(vb, bias + 128, extra ? extra + 128 : 0u, nullptr, hb, lo);
#pragma unroll
  for (int j = 0; j < 16; ++j) { h[j] = ha[j]; h[16 + j] = hb[j]; }
}
__device__ __forceinline__ void store32(uint32_t t_p, const uint32_t (&h)[32]) {
  uint32_t a[16], b[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) { a[j] = h[j]; b[j] = h[16 + j]; }
  tmem_st16(t_p, a);
  tmem_st16(t_p + 16, b);
}

// Epilogue of half h of step s of one stream for this thread's row (its TMEM lane) and columns [64 ch, 64 ch + 64).  t_p / t_q:
// the stream's operand P / accumulator Q at this lane; gate: the stream's gate barrier; bias: the step's bias block.  A half-0 result is HELD in `keep` until
// half 1, when P is dead.  Step 6 adds the per-ray direction term dir_row (of the row's ray rp) and leaves sigma's raw value in
// sigma_raw; step 9 turns it and the colour into what compositing needs -> *pre (live rows; dbg_raw, when not null, gets the raw
// outputs).  Signals the gate once Q has been read (and P holds the next operand), except after the last step.
__device__ __forceinline__ void epilogue_event(const RenderParams& p, int s, int h, uint32_t t_p, uint32_t t_q, uint32_t gate,
                                               const float* bias, const float* dir_row, uint32_t (&keep)[32], float& sigma_raw,
                                               const RayP& rp, bool has_bg, bool live, int pass, int S, int i, int ch, int lane,
                                               float4* pre, float* dbg_raw) {
  const int c0 = 64 * ch;
  uint32_t hh[32];
  bool arrived = false;
  if (s <= 5) {
    if (h == 0) {  // outputs [64 ch, +64) of features 0..127 -> registers (gate signalled inside)
      epi_load64_early(t_q + c0, smem_u32(bias + c0), 0u, keep, gate, lane);
      arrived = true;
    } else {       // P is dead: store half 0 (K atom ch), convert half 1 (K atom 2 + ch)
      store32(t_p + 32 * ch, keep);
      epi_load64(t_q + c0, smem_u32(bias + 128 + c0), 0u, hh);
      store32(t_p + 64 + 32 * ch, hh);
      tmem_wait_st();
    }
  } else if (s == 6) {
    if (h == 0) {
      epi_load64_early(t_q + c0, smem_u32(bias + c0), smem_u32(dir_row + c0), keep, gate, lane);
      arrived = true;
    } else {  // sigma = column 0 of the 16-wide second half; then g0 becomes the operand (K = 128)
      if (ch == 0) {
        uint32_t v[4];
        tmem_ld4(t_q, v);
        tmem_wait_ld();
        sigma_raw = __uint_as_float(v[0]) + bias[128];
      }
      store32(t_p + 32 * ch, keep);
      tmem_wait_st();
    }
  } else if (s <= 8) {  // 128 -> 128 layers: the MMAs that read P have completed
    epi_load64(t_q + c0, smem_u32(bias + c0), 0u, hh);
    store32(t_p + 32 * ch, hh);
    tmem_wait_st();
  } else if (ch == 0) {  // fc_rgb output
    uint32_t v[4];
    tmem_ld4(t_q, v);
    tmem_wait_ld();
    if (live) {
      const float r0 = __uint_as_float(v[0]) + bias[0], r1 = __uint_as_float(v[1]) + bias[1], r2 = __uint_as_float(v[2]) + bias[2];
      if (dbg_raw && rp.valid) reinterpret_cast<float4*>(dbg_raw)[(size_t)rp.gidx * S + i] = make_float4(r0, r1, r2, sigma_raw);
      float sig_in;
      *pre = colour_sigma(p, rp, has_bg, r0, r1, r2, sigma_raw, pass, S, i, sig_in);
    }
  }
  if (s < kNumSteps - 1 && !arrived) {
    tc_fence_before_sync();
    __syncwarp();
    if (lane == 0) mbar_arrive(gate);
  }
}

// Weight producer: the 54 loads of one tile pair from the packed stream `base` into the ring (whole warp; elected lane issues).
// `seq` counts loads across the kernel: the two CTAs of a cluster take turns issuing each load as a cluster multicast.
__device__ __forceinline__ void produce_tile(const uint8_t* __restrict__ base, uint32_t ring, uint32_t bar_full, uint32_t bar_empty,
                                             uint32_t cta_rank, uint32_t& slot, uint32_t& phase, uint32_t& seq) {
  constexpr uint16_t kAllCtas = (1u << kCluster) - 1;
  for (int i = 0; i < kNumLoads; ++i) {
    const Load& L = c_loads.l[i];
    const uint32_t piece = (uint32_t)L.rows * 128u, bytes = piece * (uint32_t)L.n_atoms;
    mbar_wait(bar_empty + slot * 8, phase ^ 1);
    if (elect_one()) {
      mbar_arrive_expect_tx(bar_full + slot * 8, bytes);
      if ((seq % kCluster) == cta_rank)
        for (int a = 0; a < L.n_atoms; ++a)
          bulk_g2s_multicast(ring + slot * kSlotBytes + a * piece, base + L.src[a], piece, bar_full + slot * 8, kAllCtas);
    }
    __syncwarp();
    ++seq;
    if (++slot == kNumSlots) { slot = 0; phase ^= 1; }
  }
}

}  // namespace t2
}  // namespace nfb
