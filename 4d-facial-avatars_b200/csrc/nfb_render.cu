// nfb_render.cu — the per-ray hot path as ONE persistent sm_100a kernel, ONE tile in flight per SM.  This is the kernel for
// exact mode (FP16 hi+lo operands), the training forward (SAVE: also writes the activation records the backward reads) and
// the debug probes; fast-mode evaluation runs the two-tiles-in-flight variant in nfb_render2.cu.
//
// Reference path replaced (nerface_code/nerf-pytorch/nerf/):
//   train_utils.py:36-162  predict_and_render_radiance   (sampling, coarse->fine control flow)
//   train_utils.py:9-33    run_network                    (encode + MLP over all samples)
//   nerf_helpers.py:195-239 positional_encoding, :344-387 sample_pdf_2, :44-65 cumprod_exclusive,
//   nerf_helpers.py:68-123 get_ray_bundle (optional in-kernel ray generation)
//   volume_rendering_utils.py:7-75 volume_render_radiance_field
//   models.py:236-261      ConditionalBlendshapePaperNeRFModel.forward
//
// Work decomposition.  A "unit of work" is R (1 or 2) rays.  One CTA per SM (clusters of 2 CTAs) loops over them;
// per ray pair it runs the coarse pass (R*Nc sample rows) and the fine pass (R*(Nc+Nf) rows) as 128-row tensor-core tiles.
// Per tile the MLP is 10 GEMM steps (nfb_layout.h).  TMEM holds two 256-column regions used alternately: step s
// accumulates (FP32) into one while its A operand — the previous step's output, converted IN PLACE to FP16 by the
// epilogue — is read from the other; hidden activations never leave TMEM.  Weights stream L2 -> shared memory through
// the bulk-copy (TMA) engine into a 5-slot ring (4 in exact mode) of pre-swizzled 32 KB units ([N rows x 64 K]); the two CTAs of a
// cluster take turns issuing each copy as a cluster multicast, so every weight byte is read from L2 once per SM pair.
// The epilogue converts and signals the accumulator in two column halves, and the units of the next step are ordered
// so that the MMAs needing only the first half are issued while the second half is still being converted.
//
// Warp roles (320 threads): warp 0 = weight producer, warp 1 = tcgen05.mma issuer (also owns the TMEM
// allocation), warps 2..9 = "row" warps.  A row warp may only touch the TMEM lane quadrant (warp & 3), so
// two warps share each quadrant: thread <-> sample row (TMEM lane), and the pair splits the columns.  They
// do sampling, positional encoding, per-step epilogues (bias, ReLU, FP16 split), compositing,
// inverse-CDF resampling and the per-ray sort.
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math_constants.h>

#include "nfb_internal.h"
#include "nfb_layout.h"
#include "nfb_ptx.cuh"
#include "nfb_save.cuh"
#include "nfb_render_common.cuh"

namespace nfb {

constexpr int kNumSlots = 5;    // ring of 32 KB weight units (exact mode uses 4: slot 4 holds the lo half of the PE operand)
constexpr int kRowsMax = 512;   // sample rows of one pass of one unit of work
constexpr int kThreads = 320;   // producer warp + MMA warp + 8 row warps
// SAVE (training forward): 512 threads — warps 0/1 producer / MMA, 2..3 idle (setmaxnreg works on whole warpgroups), 4..11 the
// row warps, 12..15 the RECORD SAVERS: one per TMEM lane quadrant, they read the FP16 activations the epilogue left in TMEM (the
// next step's A operand) and write the transposed record images — ~2,200 two-byte stores per tile and warp that used to sit on
// the row warps' critical path.  The MMA warp may not overwrite a region before its savers have read it (bar_saved).
constexpr int kThreadsSave = 512;
constexpr int kRegsLight = 80, kRegsRow = 176, kRegsSaver = 80;
static_assert((4 * kRegsLight + 8 * kRegsRow + 4 * kRegsSaver) * 32 <= 65536, "register file");
template <int N> __device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N> __device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
#ifndef NFB_CLUSTER
#define NFB_CLUSTER 2
#endif
constexpr int kCluster = NFB_CLUSTER;  // CTAs (SMs) per cluster sharing every weight unit through one multicast L2 read
constexpr int kRowThreads = 256;
constexpr uint32_t kRowBarrier = 1;  // named barrier id of the eight row warps

// TMEM column map (512 columns x 128 lanes x 32 bit): two 256-column regions used alternately.  Step s
// accumulates into region (s & 1): half 0 in its columns [0,128), half 1 in [128,256).  The epilogue converts each
// 64-column accumulator slice IN PLACE into FP16: hi part in the slice's first 32 columns (= 64 K elements = one K
// atom of the next step), lo part (exact mode) in the next 32.  Step s+1 therefore reads its A operand from
// region (s & 1) at column 64 * atom and accumulates into the other region — no separate activation buffer.
__device__ __forceinline__ uint32_t region_col(int s) { return (s & 1) ? 256u : 0u; }

// shared memory map (bytes from the 1024-aligned base)
constexpr int kOffRing = 0;
constexpr int kOffPeHi = kOffRing + kNumSlots * kMaxUnitBytes;
constexpr int kOffPeLo = kOffRing + (kNumSlots - 1) * kMaxUnitBytes;  // exact mode only: inside the last ring slot
constexpr int kOffBias = kOffPeHi + kTileM * 128;
constexpr int kOffRaw = kOffBias + 2 * kBiasFloats * 4;
constexpr int kOffZ = kOffRaw + kRowsMax * 16;
constexpr int kOffW = kOffZ + kRowsMax * 4;
constexpr int kOffCdf = kOffW + kRowsMax * 4;
constexpr int kOffBins = kOffCdf + kRowsMax * 4;
constexpr int kOffSort = kOffBins + kRowsMax * 4;
constexpr int kOffDirBias = kOffSort + kRowsMax * 4;
constexpr int kOffRay = kOffDirBias + 2 * 128 * 4;
constexpr int kOffBars = kOffRay + 2 * kRayFloats * 4;
constexpr int kNumBars = 2 * kNumSlots + 4 + 6;  // + SAVE: bar_sv[2 halves][2 step parities], bar_saved[2 regions]
constexpr int kOffTmemPtr = kOffBars + kNumBars * 8;
constexpr int kMaxProg = 40;                     // weight units per tile (32 with the current step table)
constexpr int kSmemBytes = kOffTmemPtr + 16;
static_assert(kOffBias % 16 == 0 && kOffRaw % 16 == 0 && kOffBars % 8 == 0, "alignment");

// Per-unit program entry, precomputed at compile time (the step/unit tables of nfb_layout.h involve divisions that are
// far too slow for the issue loops):  x = instruction descriptor, y = accumulator column | A column << 16 (TMEM columns
// relative to the allocation base), z = flags, w = (byte offset in the x1 weight stream) / 16 | rows << 20.
enum : uint32_t {
  kUnitFromPe = 1u, kUnitWait0 = 2u, kUnitWait1 = 4u, kUnitFirst = 8u, kUnitCommit0 = 16u, kUnitCommit1 = 32u, kUnitPostWait1 = 64u,
  kUnitStepStart = 128u,  // first unit of its step (SAVE: the accumulator region must have been read by the record savers)
  kUnitOddRegion = 256u,  // the step accumulates into region 1
  kUnitSaved = 512u       // the step's output goes to the training record (steps 0..8)
};
constexpr int total_units() {
  int n = 0;
  for (int s = 0; s < kNumSteps; ++s) n += num_units(s);
  return n;
}
constexpr int kTileUnits = total_units();
static_assert(kTileUnits <= kMaxProg, "program area too small");

struct ProgEntry { uint32_t x, y, z, w; };
struct ProgTable { ProgEntry e[kMaxProg]; };
constexpr uint32_t region_col_c(int s) { return (s & 1) ? 256u : 0u; }
constexpr ProgTable make_prog() {
  ProgTable t{};
  int i = 0;
  for (int s = 0; s < kNumSteps; ++s) {
    const StepInfo si = step_info(s);
    const int nu = num_units(s);
    bool any_g2 = false;
    for (int j = 0; j < nu; ++j) any_g2 = any_g2 || unit_info(s, j).group == 2;
    for (int u = 0; u < nu; ++u, ++i) {
      const UnitInfo ui = unit_info(s, u);
      bool first_of_half = true, first_g1 = true, first_g2 = true;
      for (int j = 0; j < u; ++j) {
        const UnitInfo uj = unit_info(s, j);
        if (uj.h == ui.h) first_of_half = false;
        if (uj.group == 1) first_g1 = false;
        if (uj.group == 2) first_g2 = false;
      }
      uint32_t flags = 0;
      if (ui.from_pe) flags |= kUnitFromPe;
      if (ui.group == 1 && first_g1) flags |= kUnitWait0;
      if (ui.group == 2 && first_g2) flags |= kUnitWait1;
      if (first_of_half) flags |= kUnitFirst;
      if (ui.last) flags |= kUnitCommit0;                               // the step's accumulator is complete
      if (u == 0) flags |= kUnitStepStart;
      if (s & 1) flags |= kUnitOddRegion;
      if (s <= 8) flags |= kUnitSaved;
      if (u == nu - 1 && !any_g2) flags |= kUnitPostWait1;           // still consume the half-1 "converted" signal
      const uint32_t d_col = region_col_c(s);
      const uint32_t a_col = (region_col_c(s) ^ 256u) + (uint32_t)(ui.ka - si.pe_first) * 64u;
      t.e[i].x = umma_idesc_f16(kTileM, ui.rows);
      t.e[i].y = d_col | (a_col << 16);
      t.e[i].z = flags;
      t.e[i].w = ((uint32_t)(step_offset_x1(s) + unit_offset_in_step(s, u)) >> 4) | ((uint32_t)ui.rows << 20);  // rows <= 256
    }
  }
  return t;
}
// Constant memory: the issue loops index it with a warp-uniform counter, so entries arrive in uniform registers
// (ULDC) — which is where UTCHMMA / UBLKCP take their operands from.  (From shared memory every field needs an R2UR.)
__constant__ ProgTable c_prog = make_prog();
static_assert(kSmemBytes <= 232448, "exceeds the 227 KB per-CTA shared memory limit");

// Epilogue of one 64-column accumulator slice (this thread's share of one N-half): both TMEM loads in flight,
// two independent bias/ReLU/convert chains, then the FP16 result overwrites the slice in place — hi in columns
// [0,32), lo (exact mode) in [32,64).  All reads complete (wait::ld) before the first store.
//
// The FP16 (hi) values are handed back: the training forward (SAVE) writes them, and the ReLU mask derived from them,
// to the tile record AFTER it has signalled the gate, so that work overlaps the next step's tensor-core time.
template <bool EXACT>
__device__ __forceinline__ void epi_half(uint32_t t_slice, uint32_t bias, uint32_t extra, float* __restrict__ dump,
                                         uint32_t (&ha)[16], uint32_t (&hb)[16]) {
  uint32_t va[32], vb[32], la[16], lb[16];
  tmem_ld32(t_slice, va);
  tmem_ld32(t_slice + 32, vb);
  tmem_wait_ld();
  epi_math<EXACT>(va, bias, extra, dump, ha, la);
  epi_math<EXACT>(vb, bias + 128, extra ? extra + 128 : 0u, dump ? dump + 32 : nullptr, hb, lb);
  tmem_st16(t_slice, ha);
  tmem_st16(t_slice + 16, hb);
  if constexpr (EXACT) {
    tmem_st16(t_slice + 32, la);
    tmem_st16(t_slice + 48, lb);
  }
}

// ------------------------------------------------------------------------------------------------
// LO (the exact-gradient training forward, EXACT and SAVE only): the records are 2 MiB and the lo parts of every image go to the
// second MiB (nfb_layout.h kRecLo) — the savers read the lo columns (+32 of each slice) too, the row warps write the lo PE and PEd
// images.
template <bool EXACT, bool SAVE, bool LO = false>
__global__ void __launch_bounds__(SAVE ? kThreadsSave : kThreads, 1) render_kernel(const __grid_constant__ RenderParams p) {
  static_assert(!LO || (EXACT && SAVE), "lo records need the exact training forward");
  constexpr long long kRecStride = rec_stride(LO);
  // Use the dynamic shared array directly (no integer round trip) so the compiler keeps the shared address
  // space and emits LDS/STS instead of generic loads; the swizzled operands need 1024-byte alignment.
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t smem_base = smem_u32(smem);
  if ((smem_base & 1023u) != 0u) __trap();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int NPART = EXACT ? 2 : 1;
  constexpr uint32_t NSLOT = EXACT ? kNumSlots - 1 : kNumSlots;

  const uint32_t bar_full = smem_base + kOffBars;               // [kNumSlots]
  const uint32_t bar_empty = bar_full + kNumSlots * 8;          // [kNumSlots]
  const uint32_t bar_aready = bar_empty + kNumSlots * 8;        // [2] half-h output of the previous step converted
  const uint32_t bar_accfull = bar_aready + 16;                 // [2] all MMAs of the current step completed ([0] used)
  const uint32_t bar_sv = bar_accfull + 16;                     // SAVE [half][step & 1]: the step's FP16 output is in TMEM -> savers
  const uint32_t bar_saved = bar_sv + 32;                       // SAVE [region]: the savers have read the region -> MMA warp
  constexpr int kRow0 = SAVE ? 4 : 2;                           // first of the eight row warps
  constexpr int NT = SAVE ? kThreadsSave : kThreads;
  volatile uint32_t* tmem_ptr_s = reinterpret_cast<volatile uint32_t*>(smem + kOffTmemPtr);
  float* bias_s = reinterpret_cast<float*>(smem + kOffBias);

  if (threadIdx.x == 0) {
    for (int i = 0; i < kNumSlots; ++i) {
      mbar_init(bar_full + i * 8, 1);
      mbar_init(bar_empty + i * 8, kCluster);  // released by the MMA warp of every CTA of the cluster
    }
    for (int h = 0; h < 2; ++h) {
      mbar_init(bar_aready + h * 8, kRowThreads / 32);  // one arrival per row warp per step
      mbar_init(bar_accfull + h * 8, 1);
      mbar_init(bar_sv + h * 16, kRowThreads / 32);
      mbar_init(bar_sv + h * 16 + 8, kRowThreads / 32);
      mbar_init(bar_saved + h * 8, 4);  // one arrival per saver warp
    }
    mbar_fence_init();
  }
  if (warp == 1) {
    tmem_alloc(smem_base + kOffTmemPtr, 512);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < kBiasFloats; i += NT) {
    bias_s[i] = p.bias[0][i];
    bias_s[kBiasFloats + i] = (p.nf > 0) ? p.bias[1][i] : 0.f;
  }
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();  // peer barriers are initialised before anyone multicasts into them
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr_s;
  const uint32_t cta_rank = cluster_ctarank();
  constexpr uint16_t kAllCtas = (1u << kCluster) - 1;

  // Both CTAs of a cluster run the same number of iterations (they share the weight ring protocol); a CTA
  // without a real unit in the last one renders invalid rays (no outputs).
  const int first_in_cluster = (int)blockIdx.x - (int)cta_rank_early();
  const int n_iter = (p.n_units - first_in_cluster + (int)gridDim.x - 1) / (int)gridDim.x;
  const int tiles_per_unit = p.tiles_c + p.tiles_f;

  // SAVE: every role re-partitions the register file first thing inside its own branch (whole warpgroups: 0..3, 4..11, 12..15);
  // ptxas allocates each branch against the count set there.
  if (warp == 0) {
    // ============================== weight producer ==============================
    // The whole warp runs the (warp-uniform) loop; one elected lane issues the copies.
    if constexpr (SAVE) reg_dec<kRegsLight>();
    {
      uint32_t slot = 0, phase = 0, seq = 0;
      PhaseTimer tm(p.prof, p.prof != nullptr && lane == 0);
      for (int it = 0; it < n_iter; ++it) {
        for (int t = 0; t < tiles_per_unit; ++t) {
          const uint8_t* base = p.wstream[t < p.tiles_c ? 0 : 1];
          for (int i = 0; i < kTileUnits; ++i) {
            const uint32_t w = c_prog.e[i].w;
            const uint32_t off = (w & 0xFFFFFu) << 4, bytes = (w >> 20) * 128u;
#pragma unroll
            for (int part = 0; part < NPART; ++part) {
              const uint8_t* src = EXACT ? base + 2 * (size_t)off + part * bytes : base + off;
              mbar_wait(bar_empty + slot * 8, phase ^ 1);  // slot released in every CTA of the cluster
              if (elect_one()) {
                mbar_arrive_expect_tx(bar_full + slot * 8, bytes);
                if ((seq % kCluster) == cta_rank)  // the CTAs take turns loading; every copy lands in all of them
                  bulk_g2s_multicast(smem_base + kOffRing + slot * kMaxUnitBytes, src, bytes, bar_full + slot * 8, kAllCtas);
              }
              __syncwarp();
              ++seq;
              if (++slot == NSLOT) { slot = 0; phase ^= 1; }
            }
          }
          tm.lap(41);
        }
      }
    }
  } else if (warp == 1) {
    // ============================== MMA issuer ==============================
    // Warp-uniform loop (all 32 lanes wait on the barriers); one elected lane issues tcgen05.mma / commit.
    if constexpr (SAVE) reg_dec<kRegsLight>();
    {
      uint32_t slot = 0, phase = 0, ph_a0 = 0, ph_a1 = 0;
      uint32_t sv_pending = 0, sv_phase = 0;  // SAVE, per region bit: a saved step lives there / parity of bar_saved
      PhaseTimer tm(p.prof, p.prof != nullptr && lane == 0);
      const bool prof_on = NFB_TIMERS && p.prof != nullptr;
      long long acc_gate = 0, acc_full = 0, acc_issue = 0, tq = prof_on ? clock64() : 0;
      const uint64_t pe_desc_hi = umma_smem_desc_sw128(smem_base + kOffPeHi);
      const uint64_t pe_desc_lo = umma_smem_desc_sw128(smem_base + kOffPeLo);
      for (int it = 0; it < n_iter; ++it) {
        for (int t = 0; t < tiles_per_unit; ++t) {
          for (int i = 0; i < kTileUnits; ++i) {
            const ProgEntry e = c_prog.e[i];
            if (prof_on) { const long long tn = clock64(); acc_issue += tn - tq; tq = tn; }
            if constexpr (SAVE) {
              if (e.z & kUnitStepStart) {  // this step overwrites its region: the savers must be done with what lived there
                const uint32_t rho = (e.z & kUnitOddRegion) ? 1u : 0u;
                if (sv_pending & (1u << rho)) {
                  mbar_wait(bar_saved + rho * 8, (sv_phase >> rho) & 1u);
                  sv_phase ^= 1u << rho;
                  sv_pending &= ~(1u << rho);
                  tc_fence_after_sync();
                }
                if (e.z & kUnitSaved) sv_pending |= 1u << rho;
              }
            }
            if (e.z & kUnitWait0) {  // group-1 units: previous step's half-0 output (or the PE buffer) is in place
              mbar_wait(bar_aready, ph_a0);
              ph_a0 ^= 1;
              tc_fence_after_sync();
            }
            if (e.z & kUnitWait1) {  // group-2 units: previous step's half-1 output is converted too
              mbar_wait(bar_aready + 8, ph_a1);
              ph_a1 ^= 1;
              tc_fence_after_sync();
            }
            if (prof_on) { const long long tn = clock64(); acc_gate += tn - tq; tq = tn; }
            const uint32_t d_tmem = tmem_base + (e.y & 0xFFFFu);
            const uint32_t a_tmem = tmem_base + (e.y >> 16);  // hi at +0, lo at +32 (2 fp16 per column)
            const uint32_t first = (e.z & kUnitFirst) ? 0u : 1u;
#pragma unroll
            for (int part = 0; part < NPART; ++part) {
              mbar_wait(bar_full + slot * 8, phase);
              if (prof_on) { const long long tn = clock64(); acc_full += tn - tq; tq = tn; }
              tc_fence_after_sync();
              const uint64_t b_desc = umma_smem_desc_sw128(smem_base + kOffRing + slot * kMaxUnitBytes);
              if (elect_one()) {
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                  const uint64_t bd = b_desc + (uint64_t)(ks * 2);  // +32 bytes per 16-element K step
                  const uint32_t acc_flag = (first | part | ks) ? 1u : 0u;
                  if (e.z & kUnitFromPe) {
                    umma_ss(d_tmem, pe_desc_hi + (uint64_t)(ks * 2), bd, e.x, acc_flag);
                    if (EXACT && part == 0) umma_ss(d_tmem, pe_desc_lo + (uint64_t)(ks * 2), bd, e.x, 1);
                  } else {
                    umma_ts(d_tmem, a_tmem + ks * 8, bd, e.x, acc_flag);
                    if (EXACT && part == 0) umma_ts(d_tmem, a_tmem + 32 + ks * 8, bd, e.x, 1);
                  }
                }
                umma_commit_multicast(bar_empty + slot * 8, kAllCtas);  // slot free here -> tell every loader
                if (part == NPART - 1) {
                  if (e.z & kUnitCommit0) umma_commit(bar_accfull);      // half 0 complete -> its epilogue may start
                  if (e.z & kUnitCommit1) umma_commit(bar_accfull + 8);  // half 1 complete
                }
              }
              __syncwarp();
              if (++slot == NSLOT) { slot = 0; phase ^= 1; }
            }
            if (e.z & kUnitPostWait1) {
              mbar_wait(bar_aready + 8, ph_a1);
              ph_a1 ^= 1;
            }
          }
        }
      }
      if (prof_on && lane == 0) {
        atomicAdd(p.prof + 44, (unsigned long long)acc_issue);
        atomicAdd(p.prof + 45, (unsigned long long)acc_gate);
        atomicAdd(p.prof + 46, (unsigned long long)acc_full);
      }
    }
  } else if (warp >= kRow0 && warp < kRow0 + 8) {
    // ============================== row warps ==============================
    if constexpr (SAVE) reg_inc<kRegsRow>();
    const int q = warp & 3;            // TMEM lane quadrant this warp may access
    const int row = q * 32 + lane;     // tile row == TMEM lane
    const int ch = (warp - kRow0) >> 2;  // which half of the columns this warp of the quadrant pair handles
    const int ew = warp - kRow0;       // 0..7, ray index for per-ray stages
    const int etid = ch * 128 + row;   // 0..255
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    uint8_t* pe_hi = smem + kOffPeHi;
    uint8_t* pe_lo = smem + kOffPeLo;
    float4* carry_raw = reinterpret_cast<float4*>(smem + kOffRaw);
    float* carry_z = reinterpret_cast<float*>(smem + kOffZ);
    float* scr_w = reinterpret_cast<float*>(smem + kOffW);
    float* scr_cdf = reinterpret_cast<float*>(smem + kOffCdf);
    float* scr_bins = reinterpret_cast<float*>(smem + kOffBins);
    float* scr_sort = reinterpret_cast<float*>(smem + kOffSort);
    float* dirbias = reinterpret_cast<float*>(smem + kOffDirBias);
    RayP* rayp = reinterpret_cast<RayP*>(smem + kOffRay);
    const int R = p.rays_per_unit;
    const bool has_bg = p.bg != nullptr;
    uint32_t ph_acc0 = 0;
    PhaseTimer tm(p.prof, p.prof != nullptr && etid == 0);

    for (int it = 0; it < n_iter; ++it) {
      const int unit = blockIdx.x + it * gridDim.x;
      tm.lap(39);
      // ---- per-ray constants
      if (etid < R) {
        RayP& rp = rayp[etid];
        load_ray(p, unit * R + etid, rp);
        if constexpr (SAVE) {
          if (rp.valid) p.save_dnorm[rp.gidx] = rp.dnorm;
        }
      }
      named_bar_sync(kRowBarrier, kRowThreads);
      dir_encoding(p, rayp, R, etid);
      named_bar_sync(kRowBarrier, kRowThreads);
      tm.lap(0);

      for (int pass = 0; pass < 2; ++pass) {
        if (pass == 1 && p.nf == 0) break;
        const int S = pass ? p.s_fine : p.nc;
        const int rows = R * S;
        const int n_tiles = pass ? p.tiles_f : p.tiles_c;
        const float* bias_n = bias_s + pass * kBiasFloats;

        // ---- prologue of tile t: sample depth + positional encoding -> PE buffer.  Called at the start of a pass
        //      for tile 0, and for tile t+1 from inside tile t (after step 3 released the PE buffer) so that it
        //      overlaps the tensor-core work of steps 4..9.
        auto prologue = [&](int t) {
          const int prow = t * 128 + row;
          const bool live = prow < rows;
          const int r = live ? prow / S : 0;
          const int i = live ? prow - r * S : 0;
          const RayP& rp = rayp[r];
          float z = 0.f;
          if (live) {
            if (pass == 0) {
              z = coarse_depth(p, rp, i, S);
              if (ch == 0) carry_z[prow] = z;
            } else {
              z = carry_z[prow];
            }
          }
          // positional encoding of o + d*z: 63 lanes + 1 zero pad, FP16 (hi[,lo]) into the swizzled PE buffer.
          // The two threads of a row write lanes [0,32) and [32,64) respectively.
          float f[32];
          pe_lanes<EXACT>(rp, z, ch, f);
          store_pe_row<EXACT>(f, pe_hi, pe_lo, row, ch);
          if (p.dbg_act && p.dbg_act_step == -1 && unit == 0 && pass == 0 && t == 0) {
#pragma unroll
            for (int k = 0; k < 32; ++k) p.dbg_act[row * 256 + ch * 32 + k] = f[k];
          }
          if constexpr (SAVE) {  // FP16 encoding of this tile as a transposed image (input of layers_xyz.0 / .3 in dW)
            if (unit < p.n_units) {
              uint8_t* rec = p.save_rec + (size_t)(unit * tiles_per_unit + (pass ? p.tiles_c : 0) + t) * kRecStride;
              uint32_t hh[16];
#pragma unroll
              for (int e = 0; e < 16; ++e) hh[e] = pack_f16x2(f[2 * e], f[2 * e + 1]);
              store_t32(rec + kRecPE + img_row_base(64, row), row, 32 * ch, hh);
              if constexpr (LO) {  // the remainder, rounded as store_pe_row rounds the lo operand of the forward
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                  const float2 h = unpack_f16x2(hh[e]);
                  hh[e] = pack_f16x2(f[2 * e] - h.x, f[2 * e + 1] - h.y);
                }
                store_t32(rec + kRecLo + kRecPE + img_row_base(64, row), row, 32 * ch, hh);
              }
            }
          }
          fence_proxy_async_smem();  // make the generic-proxy PE stores visible to the tensor core
        };

        prologue(0);
        named_bar_sync(kRowBarrier, kRowThreads);  // carry_z of this pass is complete (coarse: written above)
        tm.lap(2);

        for (int t = 0; t < n_tiles; ++t) {
          const int prow = t * 128 + row;  // pass-local row
          const bool live = prow < rows;
          const int r = live ? prow / S : 0;
          const int i = live ? prow - r * S : 0;
          const RayP& rp = rayp[r];
          uint8_t* rec = nullptr;  // this tile's training record (SAVE mode, real units only)
          if constexpr (SAVE) {
            if (unit < p.n_units) {
              rec = p.save_rec + (size_t)(unit * tiles_per_unit + (pass ? p.tiles_c : 0) + t) * kRecStride;
              uint32_t hh[16];  // direction encoding of this row's ray: features [16*ch, 16*ch+16) -> two 8-feature halves
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const int k = 16 * ch + 2 * e;
                const float a = (live && rp.valid && k < kDimDir) ? rp.ped[k] : 0.f;
                const float b = (live && rp.valid && k + 1 < kDimDir) ? rp.ped[k + 1] : 0.f;
                hh[e] = pack_f16x2(a, b);
              }
#pragma unroll
              for (int e = 8; e < 16; ++e) hh[e] = 0u;
              // store_t32 writes 32 features; only 16 belong to this thread, so store the first 8 words by hand
              uint8_t* img = rec + kRecPEd + img_row_base(32, row);
              const uint32_t cr = (uint32_t)((row & 63) >> 3);
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const int ka = 16 * ch + 2 * e, kb = ka + 1;
                *reinterpret_cast<uint16_t*>(img + ka * 128 + ((cr ^ (uint32_t)(ka & 7)) << 4)) = (uint16_t)(hh[e] & 0xFFFFu);
                *reinterpret_cast<uint16_t*>(img + kb * 128 + ((cr ^ (uint32_t)(kb & 7)) << 4)) = (uint16_t)(hh[e] >> 16);
              }
              if constexpr (LO) {
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                  const int ka = 16 * ch + 2 * e, kb = ka + 1;
                  const float a = (live && rp.valid && ka < kDimDir) ? rp.ped[ka] : 0.f;
                  const float b = (live && rp.valid && kb < kDimDir) ? rp.ped[kb] : 0.f;
                  const float2 h = unpack_f16x2(hh[e]);
                  const uint32_t l = pack_f16x2(a - h.x, b - h.y);
                  *reinterpret_cast<uint16_t*>(img + kRecLo + ka * 128 + ((cr ^ (uint32_t)(ka & 7)) << 4)) = (uint16_t)(l & 0xFFFFu);
                  *reinterpret_cast<uint16_t*>(img + kRecLo + kb * 128 + ((cr ^ (uint32_t)(kb & 7)) << 4)) = (uint16_t)(l >> 16);
                }
              }
            }
          }
          __syncwarp();
          if (lane == 0) {  // PE buffer of tile t is in place (fenced inside prologue): both gates of step 0
            mbar_arrive(bar_aready);
            mbar_arrive(bar_aready + 8);
          }
          if (t == 0) {
            // per-ray additive term of layers_dir.0: W[:, 256:280] . PE_dir (one output feature x ray per thread),
            // computed while the tensor core runs step 0; published by the barrier before step 6.
            const float* wt = p.wd0b_t[pass];
            const RayP& rq = rayp[ch < R ? ch : 0];
            float acc0 = 0.f;
#pragma unroll 8
            for (int j = 0; j < kDimDir; ++j) acc0 = fmaf(wt[j * 128 + row], rq.ped[j], acc0);
            dirbias[ch * 128 + row] = acc0;
            tm.lap(1);
          }

          float sigma_raw = 0.f;
          for (int s = 0; s < kNumSteps; ++s) {
            const StepInfo si = step_info(s);
            const uint32_t t_acc = t_lane + region_col(s);
            float* dump = (p.dbg_act && p.dbg_act_step == s && unit == 0 && pass == 0 && t == 0) ? p.dbg_act + row * 256 : nullptr;
            // ---------------- half 0
            mbar_wait(bar_accfull, ph_acc0);
            ph_acc0 ^= 1;
            tc_fence_after_sync();
            tm.lap(10 + s);
            uint32_t ha[16], hb[16];  // FP16 activations of this thread's slice (written to the record in SAVE mode)
            if (s <= 8) {  // ReLU layers: this thread converts output columns [64*ch, 64*ch+64) of the half in place
              const int c0 = 64 * ch;
              if (s == 6 && t == 0) named_bar_sync(kRowBarrier, kRowThreads);  // dirbias written by all threads
              const uint32_t extra = (s == 6) ? smem_u32(dirbias + r * 128 + c0) : 0u;
              epi_half<EXACT>(t_acc + c0, smem_u32(bias_n + si.bias_off + c0), extra, dump ? dump + c0 : nullptr, ha, hb);
            } else if (ch == 0) {
              // fc_rgb output.  Prepare what compositing needs per sample: colour and sigma
              // (volume_rendering_utils.py:29-33, 41-53); the exp(-sigma*delta) needs the neighbour depth and
              // stays in composite_ray.
              uint32_t v[4];
              tmem_ld4(t_acc, v);
              tmem_wait_ld();
              const float* b = bias_n + si.bias_off;
              if (live) {
                const float r0 = __uint_as_float(v[0]) + b[0], r1 = __uint_as_float(v[1]) + b[1], r2 = __uint_as_float(v[2]) + b[2];
                if (rp.valid) {
                  float* dr = pass ? p.dbg_raw_f : p.dbg_raw_c;
                  if (dr) reinterpret_cast<float4*>(dr)[(size_t)rp.gidx * S + i] = make_float4(r0, r1, r2, sigma_raw);
                }
                float sig_in;
                const float4 pre = colour_sigma(p, rp, has_bg, r0, r1, r2, sigma_raw, pass, S, i, sig_in);
                carry_raw[prow] = pre;
                if constexpr (SAVE) {  // what the compositing backward needs: colour (or bg) and the ReLU input
                  if (rp.valid) reinterpret_cast<float4*>(pass ? p.save_raw_f : p.save_raw_c)[(size_t)rp.gidx * S + i] = make_float4(pre.x, pre.y, pre.z, sig_in);
                }
              }
            }
            if (s < kNumSteps - 1) {
              tmem_wait_st();
              tc_fence_before_sync();
              __syncwarp();
              if (lane == 0) {
                mbar_arrive(bar_aready);
                if constexpr (SAVE) mbar_arrive(bar_sv + (s & 1) * 8);  // s <= 8 here: the saver warps write the image
              }
            }
            if constexpr (SAVE) {  // after the gate: the ReLU masks (the FP16 images are written by the saver warps)
              if (rec && s <= 8) {
                const int c0 = 64 * ch;
                *reinterpret_cast<uint2*>(reinterpret_cast<uint32_t*>(rec + kRecMask) + (s * 128 + row) * 8 + (c0 >> 5)) = make_uint2(relu_mask32(ha), relu_mask32(hb));
              }
            }
            tm.lap(20 + s);
            // ---------------- half 1 (same accumulator, columns [128,256))
            tm.lap(30 + (s < 8 ? s : 7));
            if (s <= 5) {
              const int c0 = 128 + 64 * ch;
              epi_half<EXACT>(t_acc + c0, smem_u32(bias_n + si.bias_off + c0), 0u, dump ? dump + c0 : nullptr, ha, hb);
            } else if (s == 6 && ch == 0) {  // sigma = first column of half 1 of the folded layers_dir.0 | fc_alpha step
              uint32_t v[4];
              tmem_ld4(t_acc + 128, v);
              tmem_wait_ld();
              sigma_raw = __uint_as_float(v[0]) + bias_n[si.bias_off + 128];
            }
            if (s < kNumSteps - 1) {
              tmem_wait_st();
              tc_fence_before_sync();
              __syncwarp();
              if (lane == 0) {
                mbar_arrive(bar_aready + 8);
                if constexpr (SAVE) { if (s <= 5) mbar_arrive(bar_sv + 16 + (s & 1) * 8); }
              }
            }
            if constexpr (SAVE) {
              if (rec && s <= 5) {
                const int c0 = 128 + 64 * ch;
                *reinterpret_cast<uint2*>(reinterpret_cast<uint32_t*>(rec + kRecMask) + (s * 128 + row) * 8 + (c0 >> 5)) = make_uint2(relu_mask32(ha), relu_mask32(hb));
              }
            }
            tm.lap(48 + s);
            if (s == 3 && t + 1 < n_tiles) {  // PE buffer is free: encode the next tile under steps 4..9
              prologue(t + 1);
              tm.lap(2);
            }
          }
        }  // tiles
        named_bar_sync(kRowBarrier, kRowThreads);
        tm.lap(3);

        // ---- debug dump of the sample depths
        {
          float* dz = pass ? p.dbg_z_f : p.dbg_z_c;
          if (dz) {
            for (int k = etid; k < rows; k += kRowThreads) {
              const int rr = k / S;
              if (rayp[rr].valid) dz[(size_t)rayp[rr].gidx * S + (k - rr * S)] = carry_z[k];
            }
          }
        }

        // ---- compositing: warp `ew` renders ray `ew`
        if (ew < R && rayp[ew].valid) {
          const RayP& rp = rayp[ew];
          const int g = rp.gidx;
          float* o_rgb = pass ? p.rgb_f : p.rgb_c;
          float* o_disp = pass ? p.disp_f : p.disp_c;
          float* o_acc = pass ? p.acc_f : p.acc_c;
          const float wl = composite_ray(carry_raw + ew * S, carry_z + ew * S, scr_w + ew * S, S, rp.dnorm, p.white_bkgd != 0,
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
        if (ew < R) build_cdf(scr_w + ew * p.nc, carry_z + ew * p.nc, scr_cdf + ew * p.nc, scr_bins + ew * p.nc, p.nc, lane);
        named_bar_sync(kRowBarrier, kRowThreads);
        tm.lap(5);
        // cat(z_coarse, z_samples) per ray into scr_sort (stride s_fine)
        const int SF = p.s_fine;
        for (int k = etid; k < R * SF; k += kRowThreads) {
          const int rr = k / SF, i = k - rr * SF;
          float val;
          if (i < p.nc) {
            val = carry_z[rr * p.nc + i];
          } else {
            const int j = i - p.nc;
            const float u = p.perturb ? (rayp[rr].valid ? p.u_rand[(size_t)rayp[rr].gidx * p.nf + j] : 0.f) : p.u_fine[j];
            val = sample_pdf(scr_cdf + rr * p.nc, scr_bins + rr * p.nc, nb, u);
          }
          scr_sort[k] = val;
        }
        named_bar_sync(kRowBarrier, kRowThreads);
        tm.lap(6);
        // ---- torch.sort(cat(z, z_samples)) (train_utils.py:126) as a rank merge
        for (int k = etid; k < R * SF; k += kRowThreads) {
          const int rr = k / SF, i = k - rr * SF;
          const float* z = scr_sort + rr * SF;
          carry_z[rr * SF + merge_rank(z, p.nc, p.nf, i)] = z[i];
        }
        named_bar_sync(kRowBarrier, kRowThreads);
        tm.lap(7);
      }  // pass
    }    // units
    tc_fence_before_sync();
  } else if (SAVE && warp >= 12) {
    // ============================== record savers (SAVE only) ==============================
    // Warp 12 + q owns TMEM lanes [32q, 32q+32).  Step s (0..8) leaves its FP16 output in place in region (s & 1): features
    // [64i, 64i+64) in the 32 columns at 64i.  bar_sv[half][s & 1] (two barriers per half, alternating by step) cannot run more than
    // one phase ahead of this warp, because the step that next completes the same barrier is s + 2, whose MMAs wait for
    // bar_saved of step s.
    reg_dec<kRegsSaver>();
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    uint32_t sv_ph = 0;  // bit (half * 2 + parity): phase of bar_sv[half][parity]
    for (int it = 0; it < n_iter; ++it) {
      const int unit = blockIdx.x + it * gridDim.x;
      for (int pass = 0; pass < 2; ++pass) {
        if (pass == 1 && p.nf == 0) break;
        const int n_tiles = pass ? p.tiles_f : p.tiles_c;
        for (int t = 0; t < n_tiles; ++t) {
          uint8_t* rec = (unit < p.n_units) ? p.save_rec + (size_t)(unit * tiles_per_unit + (pass ? p.tiles_c : 0) + t) * kRecStride : nullptr;
#pragma unroll 1
          for (int s = 0; s <= 8; ++s) {
            const uint32_t par = (uint32_t)(s & 1);
            const uint32_t t_reg = t_lane + region_col(s);
            uint8_t* img = rec ? rec + rec_x_off(s) + img_row_base(rec_width(s), row) : nullptr;
            const int n_slices = rec_width(s) >> 6;  // 64 features (32 TMEM columns) at a time
#pragma unroll 1
            for (int i = 0; i < n_slices; ++i) {
              if ((i & 1) == 0) {  // slices 0, 1 belong to output half 0, slices 2, 3 to half 1
                const int h = i >> 1;
                const uint32_t bit = 1u << (h * 2 + par);
                mbar_wait(bar_sv + h * 16 + par * 8, (sv_ph & bit) ? 1u : 0u);
                sv_ph ^= bit;
                tc_fence_after_sync();
              }
              // LO: two passes per slice (hi columns, then lo columns at +32), so the savers stay at 80 registers
#pragma unroll
              for (int part = 0; part < (LO ? 2 : 1); ++part) {
                uint32_t v[32];
                tmem_ld32(t_reg + 64 * i + 32 * part, v);
                tmem_wait_ld();
                if (i == n_slices - 1 && part == (LO ? 1 : 0)) {  // the whole region has been read: the MMA warp may overwrite it
                  tc_fence_before_sync();
                  __syncwarp();
                  if (lane == 0) mbar_arrive(bar_saved + par * 8);
                }
                if (img) {
                  uint8_t* dst = img + part * kRecLo;
                  uint32_t h0[16], h1[16];
#pragma unroll
                  for (int j = 0; j < 16; ++j) { h0[j] = v[j]; h1[j] = v[16 + j]; }
                  store_t32(dst, row, 64 * i, h0);
                  store_t32(dst, row, 64 * i + 32, h1);
                }
              }
            }
          }
        }
      }
    }
    tc_fence_before_sync();
  } else if (SAVE) {
    reg_dec<kRegsLight>();  // warps 2, 3: idle, but setmaxnreg is a warpgroup-wide instruction
  }

  __syncthreads();
  cluster_sync_all();  // no CTA leaves while its peer may still signal its barriers or write its ring
  if (warp == 1) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, 512);
  }
}

int debug_prog_v4(int index, uint32_t* out) {  // host copy of the per-tile unit program (tests)
  constexpr ProgTable t = make_prog();
  if (index < 0) return kTileUnits;
  if (index >= kTileUnits) return -1;
  out[0] = t.e[index].x; out[1] = t.e[index].y; out[2] = t.e[index].z; out[3] = t.e[index].w;
  return 4;
}

cudaError_t render_kernel_setup() {
  cudaError_t e = cudaFuncSetAttribute(render_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(render_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(render_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(render_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(render_kernel<true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
}

cudaError_t launch_render(const RenderParams& p, int precision, int num_sms, cudaStream_t st, long long* launches) {
  if (p.save_rec) {  // training forward: also writes the per-tile activation records (2: with the lo MiB)
    if (precision == 2) return launch_clustered(render_kernel<true, true, true>, p, kCluster, kThreadsSave, kSmemBytes, num_sms, st, launches);
    return precision == 1 ? launch_clustered(render_kernel<true, true>, p, kCluster, kThreadsSave, kSmemBytes, num_sms, st, launches)
                          : launch_clustered(render_kernel<false, true>, p, kCluster, kThreadsSave, kSmemBytes, num_sms, st, launches);
  }
  return precision != 0 ? launch_clustered(render_kernel<true, false>, p, kCluster, kThreads, kSmemBytes, num_sms, st, launches)
                        : launch_clustered(render_kernel<false, false>, p, kCluster, kThreads, kSmemBytes, num_sms, st, launches);
}

}  // namespace nfb
