// nfb_render3.cu — the render path with two tiles in flight per SM AND the passes of consecutive rays software-pipelined
// (fast mode, evaluation).  Same reference path, same per-tile algebra, same packed weight stream and the same half-step
// machinery as nfb_render2.cu (see its header and nfb_tile2.cuh); what changes is WHO does the work between the passes.
//
// In nfb_render2.cu the eight row warps also sample, encode, composite, resample and sort; while they do, the tensor core
// idles (measured: 5.0 k of 30.0 k cycles per 128-row tile).  Here a fourth warpgroup — the SAMPLER — owns everything that
// is not an MLP epilogue, and the tile pairs of consecutive units of work are issued in the order
//
//       C(0) | C(1) F(0,0..) | C(2) F(1,0..) | C(3) F(2,0..) | ...          C(u) = coarse pass of unit u, F(u,t) = fine tiles
//
// so that while the sampler composites / resamples / sorts unit u (which needs C(u)), the tensor core runs C(u+1), and the
// fine pass of unit u starts as soon as its first tile is encoded.  Nothing in the data path changes, so the results are
// bit-identical to nfb_render2.cu's.
//
// Warps (512 threads, register file re-partitioned with setmaxnreg):
//   0        weight producer (bulk copies into the 9-slot ring, cluster multicast)            |
//   1, 2     MMA issuers of streams X, Y (compile-time-unrolled program, nfb_tile2.cuh)       |  80 registers
//   3        idle                                                                            |
//   4..11    row warps: the 17 half-step epilogues of every tile pair, nothing else             168 registers
//   12..15   sampler: per-ray constants, stratified depths, positional encoding of EVERY tile,    96 registers
//            compositing, cdf, inverse-cdf sampling, sort, output stores
//
// Hand-offs (all mbarriers, CTA-local):  pe_ready[x] sampler -> issuer x and row warps (PE buffer x of the next job is
// encoded; per-unit constants are in place);  pe_free[x] issuer x -> sampler (step 3's MMAs have read PE buffer x);
// raw_ready[pass] row warps -> sampler (colour / sigma of every sample of the pass are in shared memory);  raw_free[pass]
// sampler -> row warps (the previous unit's values of that pass have been composited);  gate / accfull / full / empty as in
// nfb_render2.cu.  Every wait of job k depends only on jobs < k, so the schedule cannot deadlock (DESIGN.md 4c).
//
// Reference semantics (unchanged): nerf/train_utils.py:36-162, nerf_helpers.py:195-239, :344-387, volume_rendering_utils.py:7-75.
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math_constants.h>

#include "nfb_internal.h"
#include "nfb_layout.h"
#include "nfb_ptx.cuh"
#include "nfb_render_common.cuh"
#include "nfb_tile2.cuh"

namespace nfb {
namespace v7 {

using namespace t2;

constexpr int kRowsC = 128;   // sample rows of one stream in the coarse pass (R * Nc)
constexpr int kRowsF = 384;   // ... in the fine pass (R * (Nc + Nf))
constexpr int kSortMax = 768; // padded fine samples of one unit of work (2R rays x next power of two of Nf)
constexpr int kThreads = 512;
constexpr int kRowWarp0 = 4, kSamplerWarp0 = 12;
constexpr int kRowThreads = 256, kSamplerThreads = 128;
constexpr uint32_t kSamplerBarrier = 2;
constexpr int kRegsLight = 80, kRegsRow = 168, kRegsSampler = 96;
static_assert(kRegsLight + 2 * kRegsRow + kRegsSampler == 512, "the four warpgroups share the 64 K-register file");

// shared memory map
constexpr int kOffRing = 0;
constexpr int kOffPe = kOffRing + kRingBytes;                  // [2 streams][128 rows x 128 B]
constexpr int kOffBias = kOffPe + 2 * kTileM * 128;            // [2 networks][kBiasFloats]
constexpr int kOffRawC = kOffBias + 2 * kBiasFloats * 4;       // [2][kRowsC] float4 (colour, sigma) of the coarse pass
constexpr int kOffRawF = kOffRawC + 2 * kRowsC * 16;           // [2][kRowsF] float4 of the fine pass
constexpr int kOffZC = kOffRawF + 2 * kRowsF * 16;             // [2 units][2][kRowsC] depths of the coarse pass: unit u + 1's are
                                                               // drawn (for C(u+1)) before unit u's are resampled
constexpr int kOffZF = kOffZC + 2 * 2 * kRowsC * 4;                // [2][kRowsF] sorted depths of the fine pass
constexpr int kOffW = kOffZF + 2 * kRowsF * 4;                 // [2][kRowsC] compositing weights of the coarse pass
constexpr int kOffCdf = kOffW + 2 * kRowsC * 4;
constexpr int kOffBins = kOffCdf + 2 * kRowsC * 4;
constexpr int kOffSort = kOffBins + 2 * kRowsC * 4;            // [kSortMax] padded fine samples; also the fine pass's compositing scratch
static_assert(kSortMax >= 2 * kRowsF, "the fine pass's compositing weights live in the sort scratch");
constexpr int kOffDirBias = kOffSort + kSortMax * 4;           // [3][4 rays][128]: coarse network (by unit parity: C(0), C(1) are
                                                               // consecutive jobs), fine network
constexpr int kOffRay = kOffDirBias + 3 * 4 * 128 * 4;         // [3 units in flight][4 rays] RayP: unit u is set up while u - 2 is
                                                               // in its fine pass and u - 1 waits for its resampling
constexpr int kOffStage = kOffRay + 3 * 4 * kRayFloats * 4;      // [24] outputs of one pass of one unit: rgb[4][3] disp[4] acc[4] w_last[4]
constexpr int kOffBars = kOffStage + 24 * 4;
constexpr int kNumBars = 2 * kNumSlots + 12;                   // full[] empty[] gate[2] accfull[2] pefree[2] peready[2] rawready[2] rawfree[2]
constexpr int kOffTmemPtr = kOffBars + kNumBars * 8;
constexpr int kSmemBytes = kOffTmemPtr + 16;
static_assert(kOffBias % 16 == 0 && kOffRawC % 16 == 0 && kOffRawF % 16 == 0 && kOffStage % 16 == 0 && kOffBars % 8 == 0, "alignment");
static_assert(kSmemBytes <= 232448, "exceeds the 227 KB per-CTA shared memory limit");

struct JobIt {
  int n_iter, Tc, Tf, blk, pass, t;
  __host__ __device__ __forceinline__ JobIt(int n, int tc, int tf) : n_iter(n), Tc(tc), Tf(tf), blk(-1), pass(0), t(-1) {}
  __host__ __device__ __forceinline__ bool next() {
    ++t;
    for (;;) {
      if (pass == 0) {
        if (blk + 1 < n_iter && t < Tc) return true;
        pass = 1; t = 0;
      }
      if (blk >= 0 && t < Tf) return true;
      ++blk; pass = 0; t = 0;
      if (blk >= n_iter) return false;
    }
  }
  __host__ __device__ __forceinline__ int unit() const { return pass == 0 ? blk + 1 : blk; }
};

template <int N> __device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N> __device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }

// Positional encoding of sample row `row` (lane half `ch`) of tile t of one stream -> PE buffer (63 lanes + zero pad, FP16,
// 128-byte swizzled).  z comes from the stream's depth buffer; rows beyond the pass encode depth 0 of ray 0 (never read back).
__device__ __forceinline__ void encode_row(const RayP* __restrict__ rays_x /* the stream's R rays */, const float* __restrict__ z_x,
                                           uint8_t* __restrict__ pe, int t, int S, int rows, int row, int ch) {
  const int prow = t * 128 + row;
  const bool live = prow < rows;
  const int r = live ? prow / S : 0;
  const float z = live ? z_x[prow] : 0.f;
  float f[32];
  pe_lanes<false>(rays_x[r], z, ch, f);
  store_pe_row<false>(f, pe, nullptr, row, ch);
}

__global__ void __launch_bounds__(kThreads, 1) render3_kernel(const __grid_constant__ RenderParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t smem_base = smem_u32(smem);
  if ((smem_base & 1023u) != 0u) __trap();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const uint32_t bar_full = smem_base + kOffBars;            // [kNumSlots]
  const uint32_t bar_empty = bar_full + kNumSlots * 8;       // [kNumSlots]
  const uint32_t bar_gate = bar_empty + kNumSlots * 8;       // [2] stream x: operand / accumulator ready for its next half-step
  const uint32_t bar_accfull = bar_gate + 16;                // [2] stream x: half-step accumulator complete
  const uint32_t bar_pefree = bar_accfull + 16;              // [2] stream x: the MMAs reading PE buffer x (steps 0, 3) are done
  const uint32_t bar_peready = bar_pefree + 16;              // [2] stream x: the sampler has encoded the next job into it
  const uint32_t bar_rawready = bar_peready + 16;            // [2] pass: every sample's (colour, sigma) is in shared memory
  const uint32_t bar_rawfree = bar_rawready + 16;            // [2] pass: the sampler has composited the previous unit's values
  volatile uint32_t* tmem_ptr_s = reinterpret_cast<volatile uint32_t*>(smem + kOffTmemPtr);

  if (threadIdx.x == 0) {
    for (int i = 0; i < kNumSlots; ++i) {
      mbar_init(bar_full + i * 8, 1);
      mbar_init(bar_empty + i * 8, 2 * kCluster);
    }
    for (int x = 0; x < 2; ++x) {
      mbar_init(bar_gate + x * 8, kRowThreads / 32);
      mbar_init(bar_accfull + x * 8, 1);
      mbar_init(bar_pefree + x * 8, 1);
      mbar_init(bar_peready + x * 8, kSamplerThreads / 32);
      mbar_init(bar_rawready + x * 8, kRowThreads / 32);
      mbar_init(bar_rawfree + x * 8, 1);
    }
    mbar_fence_init();
  }
  if (warp == 1) {
    tmem_alloc(smem_base + kOffTmemPtr, 512);
    tmem_relinquish();
  }
  // both networks' bias blocks stay resident (coarse and fine jobs interleave)
  for (int k = threadIdx.x; k < 2 * kBiasFloats; k += kThreads)
    reinterpret_cast<float*>(smem + kOffBias)[k] = p.bias[k / kBiasFloats][k % kBiasFloats];
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr_s;
  const uint32_t cta_rank = cluster_ctarank();

  const int first_in_cluster = (int)blockIdx.x - (int)cta_rank;
  const int n_iter = (p.n_units - first_in_cluster + (int)gridDim.x - 1) / (int)gridDim.x;  // units of work (2R rays) of this CTA
  const int Tc = p.tiles_c, Tf = p.tiles_f;

  // The job sequence every role walks (JobIt):  block b = -1: C(0);  block b >= 0: C(b+1) (if it exists), then F(b, 0..Tf-1).
  // A job is (u = the unit's iteration index, pass 0/1, t = tile pair of the pass).

  if (warp < kRowWarp0) {
    reg_dec<kRegsLight>();
    if (warp == 0) {
      // ============================== weight producer ==============================
      uint32_t slot = 0, phase = 0, seq = 0;
      for (JobIt j(n_iter, Tc, Tf); j.next();)
        produce_tile(p.wstream[j.pass], smem_base + kOffRing, bar_full, bar_empty, cta_rank, slot, phase, seq);
    } else if (warp <= 2) {
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
      auto group = [&](auto G) {
        constexpr int g = decltype(G)::value;
        mbar_wait(gate, ph_gate);  // operand P_x in place, accumulator Q_x read
        ph_gate ^= 1;
        tc_fence_after_sync();
        issue_loads<kLoads.gfirst[g], kLoads.gcount[g]>(c);
        if constexpr (g == kLastPeGroup) {  // step 3's second half issued: nothing reads PE buffer x after these MMAs
          if (elect_one()) umma_commit(bar_pefree + x * 8);
          __syncwarp();
        }
      };
      for (JobIt j(n_iter, Tc, Tf); j.next();) {
        mbar_wait(bar_peready + x * 8, ph_per);  // the sampler has encoded this job into PE buffer x
        ph_per ^= 1;
        for_each_group(group, std::make_integer_sequence<int, kNumGroups>{});
      }
    }
  } else if (warp < kSamplerWarp0) {
    // ============================== row warps: the half-step epilogues ==============================
    reg_inc<kRegsRow>();
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int ch = (warp - kRowWarp0) >> 2;
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    const RayP* rayp_all = reinterpret_cast<const RayP*>(smem + kOffRay);
    const int R = p.rays_per_unit;
    const bool has_bg = p.bg != nullptr;
    uint32_t ph_acc0 = 0, ph_acc1 = 0, ph_per = 0, ph_rawfree0 = 0, ph_rawfree1 = 0;

    auto job = [&](int u, int pass, int t) {
      const int S = pass ? p.s_fine : p.nc;
      const int rows = R * S;
      const int n_tiles = pass ? Tf : Tc;
      const int prow = t * 128 + row;
      const bool live = prow < rows;
      const int r = live ? prow / S : 0;
      const int i = live ? prow - r * S : 0;
      const RayP* rayp = rayp_all + (u % 3) * 4;
      const float* bias_n = reinterpret_cast<const float*>(smem + kOffBias) + pass * kBiasFloats;
      const float* dirbias = reinterpret_cast<const float*>(smem + kOffDirBias) + (pass ? 2 : (u & 1)) * 512;
      float4* raw = reinterpret_cast<float4*>(smem + (pass ? kOffRawF : kOffRawC));
      const int raw_stride = pass ? kRowsF : kRowsC;
      __syncwarp();
      if (lane == 0) {  // the previous job's accumulators have been read: the first half-steps of both streams may start
        mbar_arrive(bar_gate);
        mbar_arrive(bar_gate + 8);
      }
      // per-unit constants (rays, direction terms) written by the sampler before it signalled this job's PE buffers
      mbar_wait(bar_peready, ph_per);
      mbar_wait(bar_peready + 8, ph_per);
      ph_per ^= 1;

      uint32_t keep0[32], keep1[32];  // half-0 results of streams X / Y, held until P is dead
      float sigma_raw0 = 0.f, sigma_raw1 = 0.f;
      for (int s = 0; s < kNumSteps; ++s) {
        const float* bias_s = bias_n + step_info(s).bias_off;
        if (s == kNumSteps - 1 && t == 0) {  // about to overwrite the pass's (colour, sigma) buffer: previous unit composited?
          if (pass == 0) { mbar_wait(bar_rawfree, ph_rawfree0 ^ 1); ph_rawfree0 ^= 1; }
          else           { mbar_wait(bar_rawfree + 8, ph_rawfree1 ^ 1); ph_rawfree1 ^= 1; }
        }
        for (int h = 0; h < num_halves(s); ++h) {
#pragma unroll
          for (int x = 0; x < 2; ++x) {
            const uint32_t t_p = t_lane + (uint32_t)x * 256u;
            if (x == 0) { mbar_wait(bar_accfull, ph_acc0); ph_acc0 ^= 1; }
            else        { mbar_wait(bar_accfull + 8, ph_acc1); ph_acc1 ^= 1; }
            tc_fence_after_sync();
            epilogue_event(p, s, h, t_p, t_p + 128u, bar_gate + x * 8, bias_s, dirbias + (x * R + r) * 128, x ? keep1 : keep0,
                           x ? sigma_raw1 : sigma_raw0, rayp[x * R + r], has_bg, live, pass, S, i, ch, lane, raw + x * raw_stride + prow,
                           nullptr);
          }
        }
      }
      if (t == n_tiles - 1) {  // the pass is complete: its samples may be composited
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_rawready + pass * 8);
      }
    };
    for (JobIt j(n_iter, Tc, Tf); j.next();) job(j.unit(), j.pass, j.t);
    tc_fence_before_sync();
  } else {
    // ============================== sampler ==============================
    reg_dec<kRegsSampler>();
    const int sw = warp - kSamplerWarp0;          // 0..3
    const int stid = sw * 32 + lane;              // 0..127
    RayP* rayp_all = reinterpret_cast<RayP*>(smem + kOffRay);
    float* zc_all = reinterpret_cast<float*>(smem + kOffZC);
    float* zf = reinterpret_cast<float*>(smem + kOffZF);
    float* scr_w = reinterpret_cast<float*>(smem + kOffW);
    float* scr_cdf = reinterpret_cast<float*>(smem + kOffCdf);
    float* scr_bins = reinterpret_cast<float*>(smem + kOffBins);
    float* scr_sort = reinterpret_cast<float*>(smem + kOffSort);
    float* dirbias = reinterpret_cast<float*>(smem + kOffDirBias);
    const float4* raw_c = reinterpret_cast<const float4*>(smem + kOffRawC);
    const float4* raw_f = reinterpret_cast<const float4*>(smem + kOffRawF);
    const int R = p.rays_per_unit, RR = 2 * R;
    const int nc = p.nc, nf = p.nf, SF = p.s_fine;
    int P2 = 1;                                   // fine samples of one ray padded to a power of two for the bitonic network
    while (P2 < nf) P2 <<= 1;
    uint32_t ph_pefree = 1;                       // first wait passes: nothing has read the PE buffers yet
    uint32_t ph_rawready0 = 0, ph_rawready1 = 0;
    auto sbar = [&]() { named_bar_sync(kSamplerBarrier, kSamplerThreads); };

    // ---- per-ray constants of unit iteration `it` (ray slot e = x * R + r) and the coarse network's direction term
    auto ray_setup = [&](int it) {
      RayP* rayp = rayp_all + (it % 3) * 4;
      const int unit = blockIdx.x + it * gridDim.x;
      if (stid < RR) load_ray(p, unit * RR + stid, rayp[stid]);
      sbar();
      dir_encoding(p, rayp, RR, stid);
      sbar();
    };
    // per-ray additive term of layers_dir.0 of network `pass`: W[:, 256:280] . PE_dir; thread = output feature
    auto dir_term = [&](int it, int pass) {
      const RayP* rayp = rayp_all + (it % 3) * 4;
      const float* wt = p.wd0b_t[pass];
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
      for (int j = 0; j < kDimDir; ++j) {
        const float w = wt[j * 128 + stid];
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[e] = fmaf(w, rayp[e < RR ? e : 0].ped[j], acc[e]);
      }
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if (e < RR) dirbias[(pass ? 2 : (it & 1)) * 512 + e * 128 + stid] = acc[e];
    };
    // stratified depths of the coarse pass (train_utils.py:56-76)
    auto z_coarse = [&](int it) {
      const RayP* rayp = rayp_all + (it % 3) * 4;
      float* zc = zc_all + (it & 1) * (2 * kRowsC);
      for (int k = stid; k < RR * nc; k += kSamplerThreads) {
        const int e = k / nc, i = k - e * nc;
        const int x = e / R, rr = e - x * R;
        zc[x * kRowsC + rr * nc + i] = coarse_depth(p, rayp[e], i, nc);
      }
    };
    // positional encoding of tile t of `pass` of both streams into the PE buffers, each after its previous reader is done
    auto encode = [&](int it, int pass, int t) {
      const RayP* rayp = rayp_all + (it % 3) * 4;
      const float* zc = zc_all + (it & 1) * (2 * kRowsC);
      const int S = pass ? SF : nc, rows = R * S;
#pragma unroll
      for (int x = 0; x < 2; ++x) {
        mbar_wait(bar_pefree + x * 8, ph_pefree);
        const float* z_x = pass ? zf + x * kRowsF : zc + x * kRowsC;
        uint8_t* pe = smem + kOffPe + x * (kTileM * 128);
        for (int k = 0; k < 2; ++k) {  // 128 rows x 2 lane halves = 256 thread-tasks for 128 threads
          const int idx = k * kSamplerThreads + stid;
          encode_row(rayp + x * R, z_x, pe, t, S, rows, idx & 127, idx >> 7);
        }
        fence_proxy_async_smem();  // generic-proxy stores -> visible to the tensor core's async-proxy reads
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_peready + x * 8);
      }
      ph_pefree ^= 1;
    };
    // compositing of one pass of unit `it`: warp sw renders ray slot sw (and sw + 4 never exists: RR <= 4)
    // Compositing of one pass of unit `it`: warp sw renders ray slot sw into the staging block; store_outputs() then writes the
    // unit's results with 16-byte stores (the 2R rays of a unit are consecutive in every output array).
    float* stage = reinterpret_cast<float*>(smem + kOffStage);
    auto composite_pass = [&](int it, int pass) {
      const RayP* rayp = rayp_all + (it % 3) * 4;
      const float* zc = zc_all + (it & 1) * (2 * kRowsC);
      const int S = pass ? SF : nc;
      if (sw < RR && rayp[sw].valid) {
        const RayP& rp = rayp[sw];
        const int x = sw / R, rr = sw - x * R;
        const float4* raw = (pass ? raw_f + x * kRowsF : raw_c + x * kRowsC) + rr * S;
        const float* z = (pass ? zf + x * kRowsF : zc + x * kRowsC) + rr * S;
        float* wbuf = (pass ? scr_sort + x * kRowsF : scr_w + x * kRowsC) + rr * S;
        const float wl = composite_ray(raw, z, wbuf, S, rp.dnorm, p.white_bkgd != 0, stage + 3 * sw, stage + 12 + sw, stage + 16 + sw, lane);
        if (lane == 0) stage[20 + sw] = wl;
      }
    };
    // after a sampler barrier: the staged outputs of unit `it` -> global memory.  Full unit of 4 valid rays: float4 stores
    // (rgb: 3 per unit at 48-byte stride, the scalars 1 each); otherwise (last unit, R = 1) per-ray scalar stores.
    auto store_outputs = [&](int it, int pass) {
      const RayP* rayp = rayp_all + (it % 3) * 4;
      float* o_rgb = pass ? p.rgb_f : p.rgb_c;
      float* o_disp = pass ? p.disp_f : p.disp_c;
      float* o_acc = pass ? p.acc_f : p.acc_c;
      float* o_wl = (pass == 1) ? p.w_last : nullptr;
      const int g0 = rayp[0].gidx;
      const bool vec = (RR == 4) && rayp[3].valid;
      if (vec) {
        if (stid < 3 && o_rgb) reinterpret_cast<float4*>(o_rgb + 3 * (size_t)g0)[stid] = reinterpret_cast<const float4*>(stage)[stid];
        else if (stid == 3 && o_disp) *reinterpret_cast<float4*>(o_disp + g0) = reinterpret_cast<const float4*>(stage)[3];
        else if (stid == 4 && o_acc) *reinterpret_cast<float4*>(o_acc + g0) = reinterpret_cast<const float4*>(stage)[4];
        else if (stid == 5 && o_wl) *reinterpret_cast<float4*>(o_wl + g0) = reinterpret_cast<const float4*>(stage)[5];
      } else if (stid < RR && rayp[stid].valid) {
        const int g = rayp[stid].gidx;
        if (o_rgb) { o_rgb[3 * (size_t)g] = stage[3 * stid]; o_rgb[3 * (size_t)g + 1] = stage[3 * stid + 1]; o_rgb[3 * (size_t)g + 2] = stage[3 * stid + 2]; }
        if (o_disp) o_disp[g] = stage[12 + stid];
        if (o_acc) o_acc[g] = stage[16 + stid];
        if (o_wl) o_wl[g] = stage[20 + stid];
      }
    };
    // everything between the passes of unit `it`: composite the coarse pass, resample, sort -> zf
    auto between_passes = [&](int it) {
      const RayP* rayp = rayp_all + (it % 3) * 4;
      const float* zc = zc_all + (it & 1) * (2 * kRowsC);
      mbar_wait(bar_rawready, ph_rawready0);  // C(it) complete
      ph_rawready0 ^= 1;
      composite_pass(it, 0);
      // ---- inverse-CDF resampling (nerf_helpers.py:344-387) on weights[1:-1] over the mid-point bins
      __syncwarp();
      const int nb = nc - 1;
      if (sw < RR) {
        const int x = sw / R, rr = sw - x * R;
        const int base = x * kRowsC + rr * nc;
        build_cdf(scr_w + base, zc + base, scr_cdf + base, scr_bins + base, nc, lane);
      }
      sbar();
      if (stid == 0) mbar_arrive(bar_rawfree);  // the coarse (colour, sigma) buffer may be overwritten by C(it + 1)
      store_outputs(it, 0);
      // fine samples of every ray into scr_sort[e * P2 + j], padded with +inf
      for (int k = stid; k < RR * P2; k += kSamplerThreads) {
        const int e = k / P2, j = k - e * P2;
        float val = CUDART_INF_F;
        if (j < nf) {
          const int x = e / R, rr = e - x * R;
          const float u = p.perturb ? (rayp[e].valid ? p.u_rand[(size_t)rayp[e].gidx * nf + j] : 0.f) : p.u_fine[j];
          val = sample_pdf(scr_cdf + x * kRowsC + rr * nc, scr_bins + x * kRowsC + rr * nc, nb, u);
        }
        scr_sort[k] = val;
      }
      sbar();
      // ---- torch.sort(cat(z, z_samples)) (train_utils.py:126): bitonic network over each ray's samples, then a merge with the
      // (already increasing) coarse depths by rank.  Only the sorted VALUES are used downstream, so any correct sort is exact.
      const int n_pairs = RR * P2 / 2;
      for (int kk = 2; kk <= P2; kk <<= 1) {
        for (int jj = kk >> 1; jj > 0; jj >>= 1) {
          for (int q = stid; q < n_pairs; q += kSamplerThreads) {
            const int i = 2 * q - (q & (jj - 1));  // lower index of the q-th pair at distance jj (segments of P2 never mix: jj < P2)
            const int l = i + jj;
            const bool up = ((i & kk) == 0) || kk == P2;
            const float a = scr_sort[i], b = scr_sort[l];
            if ((a > b) == up) { scr_sort[i] = b; scr_sort[l] = a; }
          }
          sbar();
        }
      }
      for (int k = stid; k < RR * SF; k += kSamplerThreads) {
        const int e = k / SF, i = k - e * SF;
        const int x = e / R, rr = e - x * R;
        const float* zcr = zc + x * kRowsC + rr * nc;
        const float* zs = scr_sort + e * P2;
        float v;
        int rank;
        if (i < nc) {       // coarse sample: its index + the fine samples strictly below it
          v = zcr[i];
          int lo = 0, hi = nf;
          while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (zs[mid] < v) lo = mid + 1; else hi = mid;
          }
          rank = i + lo;
        } else {            // fine sample: its index + the coarse samples at or below it
          const int j = i - nc;
          v = zs[j];
          int lo = 0, hi = nc;
          while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (zcr[mid] <= v) lo = mid + 1; else hi = mid;
          }
          rank = j + lo;
        }
        zf[x * kRowsF + rr * SF + rank] = v;
      }
      sbar();
    };
    auto finish_fine = [&](int it) {  // F(it) complete -> composite it, then its buffers are free
      mbar_wait(bar_rawready + 8, ph_rawready1);
      ph_rawready1 ^= 1;
      composite_pass(it, 1);
      sbar();
      if (stid == 0) mbar_arrive(bar_rawfree + 8);
      store_outputs(it, 1);
      sbar();  // the staging block is reused by the next pass's compositing
    };

    auto prepare = [&](int u, int pass, int t) {
      if (pass == 0) {
        if (t == 0) {
          ray_setup(u);
          dir_term(u, 0);   // into the buffer of this unit's parity: C(u - 1) may still be running (C(0), C(1) are adjacent)
          z_coarse(u);
          sbar();
        }
      } else if (t == 0) {
        if (u > 0) finish_fine(u - 1);  // before zf / the fine direction terms are overwritten
        between_passes(u);
        dir_term(u, 1);
        sbar();
      }
      encode(u, pass, t);
    };
    for (JobIt j(n_iter, Tc, Tf); j.next();) prepare(j.unit(), j.pass, j.t);
    finish_fine(n_iter - 1);
  }

  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace v7

// host copy of the pipelined kernel's job sequence (tests): job `index` of a CTA with n_iter units, Tc / Tf tile pairs per pass ->
// (unit iteration, pass, tile); index < 0: the number of jobs; also the kernel's shared-memory size and per-stream row limits
int debug_jobs_v7(int n_iter, int tc, int tf, int index, uint32_t* out) {
  int k = 0;
  for (v7::JobIt j(n_iter, tc, tf); j.next(); ++k)
    if (k == index) {
      out[0] = (uint32_t)j.unit(); out[1] = (uint32_t)j.pass; out[2] = (uint32_t)j.t;
      out[3] = (uint32_t)v7::kSmemBytes; out[4] = (uint32_t)v7::kRowsC; out[5] = (uint32_t)v7::kRowsF; out[6] = (uint32_t)v7::kSortMax;
      return 7;
    }
  return index < 0 ? k : -1;
}

cudaError_t render3_kernel_setup() {
  return cudaFuncSetAttribute(v7::render3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, v7::kSmemBytes);
}

// Configurations the pipelined kernel's fixed shared-memory budget covers (nfb_api.cu falls back to nfb_render2.cu otherwise).
// It has no training variant and none of the debug outputs.
bool render3_supports(const RenderParams& p) {
  if (p.nf <= 0 || p.nc < 3 || p.save_rec) return false;
  const int R = p.rays_per_unit;
  int p2 = 1;
  while (p2 < p.nf) p2 <<= 1;
  const bool fits = R * p.nc <= v7::kRowsC && R * p.s_fine <= v7::kRowsF && 2 * R * p2 <= v7::kSortMax && !p.dbg_act && !p.prof;
  return fits && !p.dbg_z_c && !p.dbg_raw_c && !p.dbg_z_f && !p.dbg_raw_f;
}

// `p` is prepared for the one-tile kernel (n_units = units of R rays); here a unit of work is 2R rays.
cudaError_t launch_render3(const RenderParams& p_in, int num_sms, cudaStream_t st, long long* launches) {
  RenderParams p = p_in;
  p.n_units = (p_in.n_rays + 2 * p_in.rays_per_unit - 1) / (2 * p_in.rays_per_unit);
  return launch_clustered(v7::render3_kernel, p, t2::kCluster, v7::kThreads, v7::kSmemBytes, num_sms, st, launches);
}

}  // namespace nfb
