// nfb_render2.cu — the render path with TWO tiles in flight per SM (fast mode, evaluation).
//
// Same reference path and same per-tile algebra as nfb_render.cu (see its header for the reference citations); what
// changes is how the tensor core is kept busy.  With one tile per SM the epilogue -> MMA hand-off of every step is
// exposed (the tensor pipe is busy about a third of the time).  Here every CTA runs two tile "streams" X and Y in lock
// step, and every MLP step is issued as N=128 half-steps, which the gates order as  X.h0  Y.h0  X.h1  Y.h1 :
//
//   * TMEM (512 columns): stream x owns P_x = [256x, 256x+128): the FP16 A operand (K <= 256 = 4 atoms of 32 columns) and
//     Q_x = [256x+128, 256x+256): the FP32 accumulator of one half-step (N = 128).  Both halves of a step read P_x, so
//     the half-0 result is converted to FP16 and HELD IN REGISTERS (32 per thread) until the half-1 MMAs have finished
//     reading P_x; then the epilogue of half 1 stores both halves into P_x — the operand of the next step.  No shared
//     memory is spent on activations.
//   * While the row warps convert X.h0, the tensor core runs Y.h0; while they convert Y.h0 it runs X.h1; and so on: each
//     epilogue has one half-step (16 MMAs) of the other stream to hide under.
//   * Both streams use the same weights back to back, so a weight half-unit ([128 rows x 64 K] = 16 KB, a contiguous
//     half of the unit the packed stream already holds) is loaded ONCE per tile pair: L2 -> SM weight traffic per tile
//     halves.  Ring = 10 slots x 16 KB; a slot is released (cluster-multicast commits) when both streams have used it.
//
// Warps (384 threads): 0 = weight producer; 1, 2 = MMA issuers of streams X, Y (two weight units = 8 MMAs per elected
// block); 3 = helper that encodes the NEXT fine-pass tile of both streams into the PE buffers while the current tile runs;
// 4..11 = row warps (thread <-> sample row, two warps per TMEM lane quadrant splitting the columns) serving both streams.
//
// A unit of work is 2R rays (R = 2, or 1 when one ray fills the pass): rays [0,R) form stream X, rays [R,2R) stream Y;
// sampling, compositing, inverse-CDF resampling and the sort run for all 2R rays between the passes as in nfb_render.cu.
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <type_traits>
#include <utility>

#include "nfb_internal.h"
#include "nfb_layout.h"
#include "nfb_ptx.cuh"
#include "nfb_render_common.cuh"
#include "nfb_tile2.cuh"

namespace nfb {
namespace v6 {

using namespace t2;

using Timer = PhaseTimer;

constexpr int kRowsMax = 512;  // sample rows of one pass of one stream
// Warps: 0 = weight producer, 1 / 2 = MMA issuer of stream X / Y (different SM sub-partitions; one warp issuing both streams
// in turn measured 4.37 M rays/s against 4.51 M), 3 = helper, 4..11 = row warps.  12 warps still allow 168 registers per thread.
// The helper computes the positional encoding of the NEXT fine-pass tile of both streams while the row warps run the current
// tile's epilogues (in the coarse pass the row warps do it after step 3).
constexpr int kRowWarp0 = 4;
constexpr int kThreads = (kRowWarp0 + 8) * 32;
constexpr int kRowThreads = 256;
constexpr uint32_t kRowBarrier = 1;

// shared memory map.  The between-pass scratch (weights, cdf, bins, merge buffer) aliases the two positional-encoding
// buffers: those are only read by the tensor core during a pass, the scratch only lives between passes.
constexpr int kOffRing = 0;
constexpr int kOffPe = kOffRing + kNumSlots * kSlotBytes;     // [2 streams][128 rows x 128 B]
constexpr int kOffW = kOffPe;                                 // [2][kRowsMax] floats each, inside the PE buffers
constexpr int kOffCdf = kOffW + 2 * kRowsMax * 4;
constexpr int kOffBins = kOffCdf + 2 * kRowsMax * 4;
constexpr int kOffSort = kOffBins + 2 * kRowsMax * 4;
static_assert(kOffSort + 2 * kRowsMax * 4 <= kOffPe + 2 * kTileM * 128, "scratch must fit in the PE buffers");
constexpr int kOffBias = kOffPe + 2 * kTileM * 128;           // bias block of the CURRENT pass's network
constexpr int kOffRaw = kOffBias + kBiasFloats * 4;           // [2][kRowsMax] float4
constexpr int kOffZ = kOffRaw + 2 * kRowsMax * 16;
constexpr int kOffDirBias = kOffZ + 2 * kRowsMax * 4;         // [4 rays][128]
constexpr int kOffRay = kOffDirBias + 4 * 128 * 4;
constexpr int kOffBars = kOffRay + 4 * kRayFloats * 4;
constexpr int kNumBars = 2 * kNumSlots + 8;                   // full[] empty[] gate[2] accfull[2] pefree[2] peready[2]
constexpr int kOffTmemPtr = kOffBars + kNumBars * 8;
constexpr int kSmemBytes = kOffTmemPtr + 16;
static_assert(kOffBias % 16 == 0 && kOffRaw % 16 == 0 && kOffBars % 8 == 0, "alignment");
static_assert(kSmemBytes <= 232448, "exceeds the 227 KB per-CTA shared memory limit");

// Sample depth + positional encoding of tile t of stream x -> PE buffer x (63 lanes + zero pad, FP16, swizzled).
__device__ __forceinline__ void prologue_fn(const RenderParams& p, const RayP* __restrict__ rayp, float* __restrict__ carry_z,
                                            uint8_t* __restrict__ pe_base, int x, int t, int pass, int S, int rows, int R, int row,
                                            int ch) {
  const int prow = t * 128 + row;
  const bool live = prow < rows;
  const int r = live ? prow / S : 0;
  const int i = live ? prow - r * S : 0;
  const RayP& rp = rayp[x * R + r];
  float z = 0.f;
  if (live) {
    if (pass == 0) {
      z = coarse_depth(p, rp, i, S);
      if (ch == 0) carry_z[x * kRowsMax + prow] = z;
    } else {
      z = carry_z[x * kRowsMax + prow];
    }
  }
  float f[32];
  pe_lanes<false>(rp, z, ch, f);
  store_pe_row<false>(f, pe_base + x * (kTileM * 128), nullptr, row, ch);
  fence_proxy_async_smem();
}

__global__ void __launch_bounds__(kThreads, 1) render2_kernel(const __grid_constant__ RenderParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t smem_base = smem_u32(smem);
  if ((smem_base & 1023u) != 0u) __trap();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const uint32_t bar_full = smem_base + kOffBars;            // [kNumSlots]
  const uint32_t bar_empty = bar_full + kNumSlots * 8;       // [kNumSlots]
  const uint32_t bar_gate = bar_empty + kNumSlots * 8;       // [2] stream x: operand / accumulator ready for its next half-step
  const uint32_t bar_accfull = bar_gate + 16;                // [2] stream x: half-step accumulator complete
  const uint32_t bar_pefree = bar_accfull + 16;              // [2] stream x: the MMAs reading PE buffer x (steps 0, 3) are done
  const uint32_t bar_peready = bar_pefree + 16;              // [2] stream x: the helper warp has encoded the next tile into it
  volatile uint32_t* tmem_ptr_s = reinterpret_cast<volatile uint32_t*>(smem + kOffTmemPtr);
  float* bias_s = reinterpret_cast<float*>(smem + kOffBias);

  if (threadIdx.x == 0) {
    for (int i = 0; i < kNumSlots; ++i) {
      mbar_init(bar_full + i * 8, 1);
      mbar_init(bar_empty + i * 8, 2 * kCluster);
    }
    for (int x = 0; x < 2; ++x) {
      mbar_init(bar_gate + x * 8, kRowThreads / 32);
      mbar_init(bar_accfull + x * 8, 1);
      mbar_init(bar_pefree + x * 8, 1);
      mbar_init(bar_peready + x * 8, 1);
    }
    mbar_fence_init();
  }
  if (warp == 1) {
    tmem_alloc(smem_base + kOffTmemPtr, 512);
    tmem_relinquish();
  }
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr_s;
  const uint32_t cta_rank = cluster_ctarank();

  const int first_in_cluster = (int)blockIdx.x - (int)cta_rank;
  const int n_iter = (p.n_units - first_in_cluster + (int)gridDim.x - 1) / (int)gridDim.x;  // n_units = super-units of 2R rays
  const int tiles_per_unit = p.tiles_c + p.tiles_f;  // tile PAIRS per super-unit

  if (warp == 0) {
    // ============================== weight producer ==============================
    uint32_t slot = 0, phase = 0, seq = 0;
    Timer tm(p.prof, p.prof != nullptr && lane == 0);
    for (int it = 0; it < n_iter; ++it) {
      for (int t = 0; t < tiles_per_unit; ++t) {
        const uint8_t* base = p.wstream[t < p.tiles_c ? 0 : 1];
        tm.lap(41);
        produce_tile(base, smem_base + kOffRing, bar_full, bar_empty, cta_rank, slot, phase, seq);
      }
    }
  } else if (warp == 1 || warp == 2) {
    // ============================== MMA issuer of stream x = warp - 1 ==============================
    const int x = warp - 1;
    uint32_t ph_gate = 0, ph_per = 0;
    IssueCtx c;
    c.ring = smem_base + kOffRing;
    c.ring_desc_lo = desc_lo_of(smem_base + kOffRing);
    c.p_tmem = tmem_base + (uint32_t)x * 256u;
    c.q_tmem = c.p_tmem + 128u;
    c.bar_full = bar_full;
    c.bar_empty = bar_empty;
    c.bar_accfull = bar_accfull + x * 8;
    c.pe_desc = umma_smem_desc_sw128(smem_base + kOffPe + x * (kTileM * 128));
    const uint32_t gate = bar_gate + x * 8;
    for (int it = 0; it < n_iter; ++it) {
      for (int t = 0; t < tiles_per_unit; ++t) {
        const bool fine_t = t >= p.tiles_c;  // fine-pass tiles: PE buffer handshake with the helper warp
        if (fine_t && t > p.tiles_c) {                  // its encoding was written by the helper, not by the row warps
          mbar_wait(bar_peready + x * 8, ph_per);
          ph_per ^= 1;
        }
        // one half-step group: wait until operand P_x is in place and accumulator Q_x has been read, then its loads
        auto group = [&](auto G) {
          constexpr int g = decltype(G)::value;
          mbar_wait(gate, ph_gate);
          ph_gate ^= 1;
          tc_fence_after_sync();
          issue_loads<kLoads.gfirst[g], kLoads.gcount[g]>(c);
          if constexpr (g == kLastPeGroup) {  // step 3's second half issued: nothing reads PE buffer x after these MMAs
            if (fine_t) {
              if (elect_one()) umma_commit(bar_pefree + x * 8);
              __syncwarp();
            }
          }
        };
        for_each_group(group, std::make_integer_sequence<int, kNumGroups>{});
      }
    }
  } else if (warp == 3) {
    // ============================== helper: encoding of the next fine-pass tile ==============================
    if (p.nf > 0) {
      const RayP* rayp = reinterpret_cast<const RayP*>(smem + kOffRay);
      float* carry_z = reinterpret_cast<float*>(smem + kOffZ);
      const int R = p.rays_per_unit, S = p.s_fine, rows = R * S, n_tiles = p.tiles_f;
      uint32_t ph_free0 = 0, ph_free1 = 0;
      for (int it = 0; it < n_iter; ++it) {
        for (int t = 0; t < n_tiles; ++t) {
#pragma unroll
          for (int x = 0; x < 2; ++x) {
            if (x == 0) { mbar_wait(bar_pefree, ph_free0); ph_free0 ^= 1; }
            else        { mbar_wait(bar_pefree + 8, ph_free1); ph_free1 ^= 1; }
            if (t + 1 < n_tiles) {
              for (int k = 0; k < 8; ++k) {  // 128 rows x 2 lane halves = 256 thread-tasks for 32 threads
                const int idx = k * 32 + lane;
                prologue_fn(p, rayp, carry_z, smem + kOffPe, x, t + 1, 1, S, rows, R, idx & 127, idx >> 7);
              }
              __syncwarp();  // every lane has fenced its generic-proxy stores (inside prologue_fn)
              if (lane == 0) mbar_arrive(bar_peready + x * 8);
            }
          }
        }
      }
    }
  } else if (warp >= kRowWarp0) {
    // ============================== row warps ==============================
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int ch = (warp - kRowWarp0) >> 2;
    const int ew = warp - kRowWarp0;
    const int etid = ch * 128 + row;
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    float4* carry_raw = reinterpret_cast<float4*>(smem + kOffRaw);  // [x * kRowsMax + prow]
    float* carry_z = reinterpret_cast<float*>(smem + kOffZ);
    float* scr_w = reinterpret_cast<float*>(smem + kOffW);
    float* scr_cdf = reinterpret_cast<float*>(smem + kOffCdf);
    float* scr_bins = reinterpret_cast<float*>(smem + kOffBins);
    float* scr_sort = reinterpret_cast<float*>(smem + kOffSort);
    float* dirbias = reinterpret_cast<float*>(smem + kOffDirBias);
    RayP* rayp = reinterpret_cast<RayP*>(smem + kOffRay);
    const int R = p.rays_per_unit;   // rays per stream
    const int RR = 2 * R;            // rays per unit of work
    const bool has_bg = p.bg != nullptr;
    uint32_t ph_acc0 = 0, ph_acc1 = 0;
    Timer tm(p.prof, p.prof != nullptr && etid == 0);

    for (int it = 0; it < n_iter; ++it) {
      const int unit = blockIdx.x + it * gridDim.x;
      tm.lap(39);
      if (etid < RR) load_ray(p, unit * RR + etid, rayp[etid]);  // ray slot qy = x * R + r
      named_bar_sync(kRowBarrier, kRowThreads);
      dir_encoding(p, rayp, RR, etid);
      named_bar_sync(kRowBarrier, kRowThreads);
      tm.lap(0);

      for (int pass = 0; pass < 2; ++pass) {
        if (pass == 1 && p.nf == 0) break;
        const int S = pass ? p.s_fine : p.nc;
        const int rows = R * S;  // rows of one stream in this pass
        const int n_tiles = pass ? p.tiles_f : p.tiles_c;
        const float* bias_n = bias_s;
        if (p.nf > 0 || it == 0)  // bias block of this pass's network (published by the barrier after the first prologue)
          for (int k = etid; k < kBiasFloats; k += kRowThreads) bias_s[k] = p.bias[pass][k];

        auto prologue = [&](int x, int t) { prologue_fn(p, rayp, carry_z, smem + kOffPe, x, t, pass, S, rows, R, row, ch); };

        prologue(0, 0);
        prologue(1, 0);
        named_bar_sync(kRowBarrier, kRowThreads);  // carry_z of this pass is complete
        tm.lap(2);

        for (int t = 0; t < n_tiles; ++t) {
          const int prow = t * 128 + row;
          const bool live = prow < rows;
          const int r = live ? prow / S : 0;
          const int i = live ? prow - r * S : 0;
          __syncwarp();
          if (lane == 0) {  // PE buffers of tile t are in place: first half-step of both streams may start
            mbar_arrive(bar_gate);
            mbar_arrive(bar_gate + 8);
          }
          if (t == 0) {
            // per-ray additive term of layers_dir.0: W[:, 256:280] . PE_dir; thread = (output feature `row`, rays ch and ch+2)
            const float* wt = p.wd0b_t[pass];
            float acc0 = 0.f, acc1 = 0.f;
            const RayP& ra = rayp[ch < RR ? ch : 0];
            const RayP& rb = rayp[ch + 2 < RR ? ch + 2 : 0];
#pragma unroll 8
            for (int j = 0; j < kDimDir; ++j) {
              const float w = wt[j * 128 + row];
              acc0 = fmaf(w, ra.ped[j], acc0);
              acc1 = fmaf(w, rb.ped[j], acc1);
            }
            dirbias[ch * 128 + row] = acc0;
            dirbias[(ch + 2) * 128 + row] = acc1;
            tm.lap(1);
          }

          uint32_t keep0[32], keep1[32];  // half-0 results of streams X / Y, held until P is dead
          float sigma_raw0 = 0.f, sigma_raw1 = 0.f;
          for (int s = 0; s < kNumSteps; ++s) {
            const float* bias_s = bias_n + step_info(s).bias_off;
            if (s == 6 && t == 0) named_bar_sync(kRowBarrier, kRowThreads);  // dirbias written by all threads
            for (int h = 0; h < num_halves(s); ++h) {
#pragma unroll
              for (int x = 0; x < 2; ++x) {
                const uint32_t t_p = t_lane + (uint32_t)x * 256u;
                if (x == 0) { mbar_wait(bar_accfull, ph_acc0); ph_acc0 ^= 1; }
                else        { mbar_wait(bar_accfull + 8, ph_acc1); ph_acc1 ^= 1; }
                tc_fence_after_sync();
                tm.lap(10 + s);
                epilogue_event(p, s, h, t_p, t_p + 128u, bar_gate + x * 8, bias_s, dirbias + (x * R + r) * 128, x ? keep1 : keep0,
                               x ? sigma_raw1 : sigma_raw0, rayp[x * R + r], has_bg, live, pass, S, i, ch, lane,
                               carry_raw + x * kRowsMax + prow, pass ? p.dbg_raw_f : p.dbg_raw_c);
                tm.lap(20 + s);
              }
            }
            if (s == 3 && t + 1 < n_tiles && pass == 0) {  // both PE buffers are free: encode the next tile pair under steps
                                                           // 4..9 (fine pass: the helper warp does it)
              prologue(0, t + 1);
              prologue(1, t + 1);
              tm.lap(2);
            }
          }
        }  // tile pairs
        named_bar_sync(kRowBarrier, kRowThreads);
        tm.lap(3);

        // ---- debug dump of the sample depths
        {
          float* dz = pass ? p.dbg_z_f : p.dbg_z_c;
          if (dz) {
            for (int k = etid; k < RR * S; k += kRowThreads) {
              const int qy = k / S, ii = k - qy * S;
              const int x = qy / R, rr = qy - x * R;
              if (rayp[qy].valid) dz[(size_t)rayp[qy].gidx * S + ii] = carry_z[x * kRowsMax + rr * S + ii];
            }
          }
        }

        // ---- compositing: warp `ew` renders ray slot `ew`
        if (ew < RR && rayp[ew].valid) {
          const RayP& rp = rayp[ew];
          const int g = rp.gidx;
          const int x = ew / R, rr = ew - x * R;
          const int base = x * kRowsMax + rr * S;
          float* o_rgb = pass ? p.rgb_f : p.rgb_c;
          float* o_disp = pass ? p.disp_f : p.disp_c;
          float* o_acc = pass ? p.acc_f : p.acc_c;
          const float wl = composite_ray(carry_raw + base, carry_z + base, scr_w + base, S, rp.dnorm, p.white_bkgd != 0,
                                         o_rgb ? o_rgb + 3 * (size_t)g : nullptr, o_disp ? o_disp + g : nullptr,
                                         o_acc ? o_acc + g : nullptr, lane);
          const bool last_pass = (pass == 1) || (p.nf == 0);
          if (last_pass && lane == 0 && p.w_last) p.w_last[g] = wl;
        }
        if (pass == 1 || p.nf == 0) {
          named_bar_sync(kRowBarrier, kRowThreads);  // carry buffers are reused by the next unit
          tm.lap(4);
          continue;
        }
        tm.lap(4);

        // ---- inverse-CDF resampling (nerf_helpers.py:344-387) on weights[1:-1] over the mid-point bins
        __syncwarp();
        const int nb = p.nc - 1;
        if (ew < RR) {
          const int x = ew / R, rr = ew - x * R;
          const int base = x * kRowsMax + rr * p.nc;
          build_cdf(scr_w + base, carry_z + base, scr_cdf + base, scr_bins + base, p.nc, lane);
        }
        named_bar_sync(kRowBarrier, kRowThreads);
        tm.lap(5);
        // cat(z_coarse, z_samples) per ray into scr_sort (per stream: stride s_fine)
        const int SF = p.s_fine;
        for (int k = etid; k < RR * SF; k += kRowThreads) {
          const int qy = k / SF, i = k - qy * SF;
          const int x = qy / R, rr = qy - x * R;
          float val;
          if (i < p.nc) {
            val = carry_z[x * kRowsMax + rr * p.nc + i];
          } else {
            const int j = i - p.nc;
            const float u = p.perturb ? (rayp[qy].valid ? p.u_rand[(size_t)rayp[qy].gidx * p.nf + j] : 0.f) : p.u_fine[j];
            val = sample_pdf(scr_cdf + x * kRowsMax + rr * p.nc, scr_bins + x * kRowsMax + rr * p.nc, nb, u);
          }
          scr_sort[x * kRowsMax + rr * SF + i] = val;
        }
        named_bar_sync(kRowBarrier, kRowThreads);
        tm.lap(6);
        // ---- torch.sort(cat(z, z_samples)) (train_utils.py:126) as a rank merge
        for (int k = etid; k < RR * SF; k += kRowThreads) {
          const int qy = k / SF, i = k - qy * SF;
          const int x = qy / R, rr = qy - x * R;
          const float* z = scr_sort + x * kRowsMax + rr * SF;
          carry_z[x * kRowsMax + rr * SF + merge_rank(z, p.nc, p.nf, i)] = z[i];
        }
        named_bar_sync(kRowBarrier, kRowThreads);
        tm.lap(7);
      }  // pass
    }    // units
    tc_fence_before_sync();
  }

  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace v6

int debug_prog_v6(int index, uint32_t* out) {  // host copy of the two-tile program (tests), one entry per PIECE:
  // idesc, A column (0xFFFFFFFF: PE atom), flags (1 from PE, 2 first / 4 last piece of its group), (src / 16) | rows << 20,
  // group, load index, ring slot, byte offset inside the slot
  constexpr t2::LoadTable t = t2::make_loads();
  if (index < 0) return t.n_pieces;
  if (index >= t.n_pieces) return -1;
  int k = 0;
  for (int i = 0; i < t.n; ++i) {
    const t2::Load& L = t.l[i];
    for (int a = 0; a < L.n_atoms; ++a, ++k) {
      if (k != index) continue;
      const bool g_first = (i == t.gfirst[L.group]) && a == 0;
      const bool g_last = (i == t.gfirst[L.group] + t.gcount[L.group] - 1) && a == L.n_atoms - 1;
      out[0] = umma_idesc_f16(kTileM, L.rows);
      out[1] = (uint32_t)L.a_col[a];
      out[2] = (L.a_col[a] < 0 ? 1u : 0u) | (g_first ? 2u : 0u) | (g_last ? 4u : 0u);
      out[3] = ((uint32_t)L.src[a] >> 4) | ((uint32_t)L.rows << 20);
      out[4] = (uint32_t)L.group;
      out[5] = (uint32_t)i;
      out[6] = (uint32_t)(i % t2::kNumSlots);
      out[7] = (uint32_t)(a * L.rows * 128);
      return 8;
    }
  }
  return -1;
}

cudaError_t render2_kernel_setup() {
  return cudaFuncSetAttribute(v6::render2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, v6::kSmemBytes);
}

// `p` is prepared for the one-tile kernel (n_units = units of R rays); here a unit of work is 2R rays.
cudaError_t launch_render2(const RenderParams& p_in, int num_sms, cudaStream_t st, long long* launches) {
  RenderParams p = p_in;
  p.n_units = (p_in.n_rays + 2 * p_in.rays_per_unit - 1) / (2 * p_in.rays_per_unit);
  return launch_clustered(v6::render2_kernel, p, v6::kCluster, v6::kThreads, v6::kSmemBytes, num_sms, st, launches);
}

}  // namespace nfb
