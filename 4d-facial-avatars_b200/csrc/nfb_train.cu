// nfb_train.cu — backward of the render path as hand-written sm_100a kernels.
//
// The reference has no hand-written backward: `loss.backward()` (train_transformed_rays.py:389) runs torch.autograd over
// the unfused graph of train_utils.py:36-162 / volume_rendering_utils.py:7-75 / models.py:236-261.  SURVEY.md §8 (a''')
// derives what that computes; this file implements it in four stages, all on the caller's stream:
//
//   1. composite_bwd_kernel   G = dL/d(rgb, disp, acc, w_last) per ray  ->  dL/d(rgb_raw, sigma_raw) per sample.
//                             Re-evaluates the compositing of both passes from what the training forward saved (depths,
//                             colours, ReLU input of sigma) with a division-free reverse recurrence for the transmittance
//                             term.  Also yields d fc_rgb.bias / d sigma-bias sums and the max |gradient| for the scale.
//   2. chain_kernel           dX chain of the MLP per 128-row tile on tcgen05: 9 steps with transposed weight streams,
//                             same machinery as the forward kernel (TMEM-resident activations converted in place, bulk-copy
//                             weight ring with cluster multicast, two-gate epilogue).  The epilogue applies the saved ReLU
//                             masks; four record-saver warps read every dY back from TMEM and write it as a transposed FP16
//                             image into the tile record.
//   3. dw_kernel              dW[n,k] = sum_rows dY[row,n] X[row,k] for every layer: both operands are bulk-copied from
//                             the tile records (K-major images whose K axis is the sample row) and multiplied on tcgen05
//                             (M=128 output features x N input features per job, FP32 accumulation in TMEM over all tiles
//                             of the CTA), then reduced into FP32 accumulators with red.global.add.  One launch for both
//                             networks; HBM-bound, so the job groups are laid out for L2 sharing of the input images.
//   4. finalize_kernel        un-folds the kernel's parametrisation (fc_feat pre-multiplied into fc_alpha / layers_dir.0,
//                             conditioning columns folded into biases) by the chain rule and writes the 24 used parameter
//                             gradients of each network in the reference's state_dict layout, plus d latent_code.
//
// Gradients are carried in FP16 with one power-of-two loss scale per backward call (max |d raw| -> 2^10), FP32 accumulate.
// After an NFB_PREC_EXACT_GRAD forward the chain and dW kernels run their EXACT variants instead: every operand is split
// x = hi + lo in FP16 (2 MiB records, nfb_layout.h kRecLo; hi/lo weight stream stream_bwd_x3) and multiplied as
// hi·hi + hi·lo + lo·hi, ~2^-21 relative operand error, as in the exact forward.
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "nfb_internal.h"
#include "nfb_layout.h"
#include "nfb_ptx.cuh"
#include "nfb_save.cuh"

namespace nfb {

// ================================================================================================
// 1. compositing backward (SIMT; one thread per (pass, ray))
// ================================================================================================
// One WARP per (ray, pass); samples are lane-blocked (lane l owns samples [l*per, (l+1)*per)).  The forward product of
// (1 - alpha + 1e-10) and the reverse affine recurrence  C_{i-1} = dLdw_i alpha_i + omega_i C_i  are both scans: in-lane
// sequential, across lanes a shuffle scan (of products / of composed affine maps).
__global__ void __launch_bounds__(256) composite_bwd_kernel(const CompBwdParams q) {
  const int lane = threadIdx.x & 31;
  const int idx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int npass = q.nf > 0 ? 2 : 1;
  if (idx >= npass * q.n_rays) return;  // whole warps
  const int pass = idx / q.n_rays;
  const int g = idx - pass * q.n_rays;
  const int S = pass ? q.s_fine : q.nc;
  const float* __restrict__ z = (pass ? q.z_f : q.z_c) + (size_t)g * S;
  const float4* __restrict__ raw = reinterpret_cast<const float4*>(pass ? q.raw_f : q.raw_c) + (size_t)g * S;
  const float dn = q.dnorm[g];
  float G0 = 0.f, G1 = 0.f, G2 = 0.f;
  if (q.g_rgb[pass]) { G0 = q.g_rgb[pass][3 * g]; G1 = q.g_rgb[pass][3 * g + 1]; G2 = q.g_rgb[pass][3 * g + 2]; }
  const float gdisp = q.g_disp[pass] ? q.g_disp[pass][g] : 0.f;
  float g_acc = q.g_acc[pass] ? q.g_acc[pass][g] : 0.f;
  const float gwl = (pass == npass - 1 && q.g_wlast) ? q.g_wlast[g] : 0.f;
  constexpr int kPer = 16;  // S <= 512
  const int per = (S + 31) >> 5;
  const int i0 = lane * per;

  // ---- forward: alpha, e = exp(-sigma delta) per sample; transmittance in front of this lane's block
  float e_[kPer], zl[kPer];
  float prod = 1.f;
#pragma unroll
  for (int j = 0; j < kPer; ++j) {
    const int i = i0 + j;
    e_[j] = 1.f; zl[j] = 0.f;
    if (j < per && i < S) {
      zl[j] = z[i];
      const float delta = ((i < S - 1) ? (z[i + 1] - zl[j]) : 1e10f) * dn;
      const float sig = fmaxf(raw[i].w, 0.f) + (i == S - 1 ? 1e-6f : 0.f);
      e_[j] = expf(-sig * delta);
      prod *= ((1.f - (1.f - e_[j])) + 1e-10f);
    }
  }
  float incl = prod;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl *= t;
  }
  float T0 = __shfl_up_sync(0xffffffffu, incl, 1);
  if (lane == 0) T0 = 1.f;
  float depth = 0.f, acc = 0.f;
  {
    float T = T0;
#pragma unroll
    for (int j = 0; j < kPer; ++j) {
      if (j < per && i0 + j < S) {
        const float alpha = 1.f - e_[j];
        const float w = alpha * T;
        depth = fmaf(w, zl[j], depth);
        acc += w;
        T *= (1.f - alpha) + 1e-10f;
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    depth += __shfl_xor_sync(0xffffffffu, depth, o);
    acc += __shfl_xor_sync(0xffffffffu, acc, o);
  }
  // disp = 1 / max(1e-10, depth / acc)  (volume_rendering_utils.py:69); rgb += 1 - acc with a white background (:71-72)
  float g_depth = 0.f;
  if (gdisp != 0.f) {
    const float qv = depth / acc;
    if (qv > 1e-10f) {
      const float dq = -gdisp / (qv * qv);
      g_depth = dq / acc;
      g_acc += -dq * depth / (acc * acc);
    }
  }
  if (q.white_bkgd) g_acc -= (G0 + G1 + G2);

  // ---- reverse sweep.  With omega_i = 1 - alpha_i + 1e-10 and C_i = sum_{k>i} dLdw_k alpha_k prod_{i<j<k} omega_j:
  //   dL/d alpha_i = T_i (dLdw_i - C_i),   C_{i-1} = dLdw_i alpha_i + omega_i C_i      (no division by omega).
  // A lane's block maps the C entering at its top sample to the C leaving below its first: C_out = A + B C_in.
  float A = 0.f, B = 1.f;
#pragma unroll
  for (int j = kPer - 1; j >= 0; --j) {
    const int i = i0 + j;
    if (j < per && i < S) {
      const float4 r4 = raw[i];
      const float dLdw = G0 * r4.x + G1 * r4.y + G2 * r4.z + g_acc + g_depth * zl[j] + (i == S - 1 ? gwl : 0.f);
      const float om = e_[j] + 1e-10f;
      A = fmaf(om, A, dLdw * (1.f - e_[j]));
      B *= om;
    }
  }
  // suffix composition over lanes 31 .. l+1 -> the C entering this lane (exclusive, from above)
  float SA = A, SB = B;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float ta = __shfl_down_sync(0xffffffffu, SA, o), tb = __shfl_down_sync(0xffffffffu, SB, o);
    if (lane + o < 32) { SA = fmaf(SB, ta, SA); SB *= tb; }  // this (lower) block applied AFTER the higher ones: A + B (ta + tb C)
  }
  float C = __shfl_down_sync(0xffffffffu, SA, 1);  // composed map of all higher lanes applied to C = 0
  if (lane == 31) C = 0.f;

  const int unit = g / q.rays_per_unit, rr = g - unit * q.rays_per_unit;
  const int tile0 = unit * (q.tiles_c + q.tiles_f) + (pass ? q.tiles_c : 0);
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f, amax = 0.f;
  // transmittance in front of each sample of this block, walking down from the block's end
  float Tj[kPer];
  {
    float T = T0;
#pragma unroll
    for (int j = 0; j < kPer; ++j) {
      Tj[j] = T;
      if (j < per && i0 + j < S) T *= (1.f - (1.f - e_[j])) + 1e-10f;
    }
  }
#pragma unroll
  for (int j = kPer - 1; j >= 0; --j) {
    const int i = i0 + j;
    if (j < per && i < S) {
      const float4 r4 = raw[i];
      const float delta = ((i < S - 1) ? (z[i + 1] - zl[j]) : 1e10f) * dn;
      const float e = e_[j];
      const float alpha = 1.f - e;
      const float Ti = Tj[j];
      const float w = alpha * Ti;
      const float dLdw = G0 * r4.x + G1 * r4.y + G2 * r4.z + g_acc + g_depth * zl[j] + (i == S - 1 ? gwl : 0.f);
      const float dalpha = Ti * (dLdw - C);
      const float dsig = dalpha * (delta * e);  // d alpha / d sigma = delta exp(-sigma delta); (1e10 * 0) stays 0
      float4 d;
      d.w = (r4.w > 0.f) ? dsig : 0.f;          // ReLU (the +1e-6 on the last sample is an additive constant)
      if (q.has_bg && i == S - 1) {
        d.x = d.y = d.z = 0.f;                  // background colour is data (train_background=False)
      } else {
        d.x = w * G0 * r4.x * (1.f - r4.x);     // sigmoid
        d.y = w * G1 * r4.y * (1.f - r4.y);
        d.z = w * G2 * r4.z * (1.f - r4.z);
      }
      C = fmaf(e + 1e-10f, C, dLdw * alpha);
      const int prow = rr * S + i;
      reinterpret_cast<float4*>(q.draw)[(size_t)(tile0 + (prow >> 7)) * 128 + (prow & 127)] = d;
      s0 += d.x; s1 += d.y; s2 += d.z; s3 += d.w;
      amax = fmaxf(amax, fmaxf(fmaxf(fabsf(d.x), fabsf(d.y)), fmaxf(fabsf(d.z), fabsf(d.w))));
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s0 += __shfl_xor_sync(0xffffffffu, s0, o); s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o); s3 += __shfl_xor_sync(0xffffffffu, s3, o);
    const float t = __shfl_xor_sync(0xffffffffu, amax, o);
    amax = (t != t || amax != amax) ? __int_as_float(0x7fc00000) : fmaxf(amax, t);
  }
  if (lane == 0) {
    float* braw = q.acc[pass] + kAccBRaw;
    atomicAdd(braw + 0, s0); atomicAdd(braw + 1, s1); atomicAdd(braw + 2, s2); atomicAdd(braw + 3, s3);
    if (amax == amax && amax < 3.0e38f) atomicMax(q.absmax, __float_as_uint(amax));
  }
}

// scal[0] = loss scale (power of two bringing max |d raw| to about 2^10), scal[1] = 1 / scale.
__global__ void scale_kernel(const unsigned int* __restrict__ absmax, float* __restrict__ scal) {
  const float m = __uint_as_float(*absmax);
  int e = 0;
  if (m > 0.f) {
    e = 10 - (int)ceilf(log2f(m));
    e = max(-100, min(100, e));
  }
  scal[0] = exp2f((float)e);
  scal[1] = exp2f((float)-e);
}

// ================================================================================================
// backward weight stream: unit (step s, K atom) = [N rows x 64 K] FP16, 128-byte swizzled, element (n, k) = W^T
// ================================================================================================
struct BwdUnit { int16_t from_op, group, rows, last, ka; };
__host__ __device__ constexpr BwdUnit bwd_unit_info(int s, int u) {
  const StepInfo si = bwd_step_info(s);
  const int hid = u - si.pe_first;
  return BwdUnit{(int16_t)(si.pe_first && u == 0), (int16_t)((hid >= 2) ? 2 : 1), (int16_t)(si.nh0 + si.nh1),
                 (int16_t)(u == si.k_atoms - 1), (int16_t)u};
}
__host__ __device__ constexpr int bwd_unit_offset(int s, int u) { return bwd_step_offset(s) + u * (bwd_step_info(s).nh0 + bwd_step_info(s).nh1) * 128; }

// (the transposed stream is written by repack_kernel, nfb_pack.cu)

// ================================================================================================
// 2. dX chain kernel
// ================================================================================================
namespace chain {

constexpr int kNumSlots = 5;
// 512 threads: warp 0 weight producer, 1 MMA issuer, 2..3 idle (setmaxnreg works on whole warpgroups), 4..11 row warps,
// 12..15 record savers — as in the training forward (nfb_render.cu), they read each step's FP16 output back from TMEM and write
// the transposed dY image, so the ~1,900 two-byte stores per tile and warp are off the row warps' critical path.
constexpr int kThreads = 512;
constexpr int kRegsLight = 80, kRegsRow = 176, kRegsSaver = 80;
static_assert((4 * kRegsLight + 8 * kRegsRow + 4 * kRegsSaver) * 32 <= 65536, "register file");
template <int N> __device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N> __device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
constexpr int kCluster = 2;
constexpr int kRowThreads = 256;
constexpr int kOffRing = 0;
constexpr int kOffOp = kOffRing + kNumSlots * kMaxUnitBytes;  // d raw operand: [128 rows x 64 k] FP16, swizzled (k < 4 used)
// EXACT (exact-gradient chain): every weight unit is loaded as two ring entries, hi then lo (stream_bwd_x3), and the d raw operand
// has a lo buffer right after the hi one.
__host__ __device__ constexpr int op_buffers(bool exact) { return exact ? 2 : 1; }
__host__ __device__ constexpr int off_bars(bool exact) { return kOffOp + op_buffers(exact) * kTileM * 128; }
constexpr int kNumBars = 2 * kNumSlots + 4 + 6;  // + bar_sv[2 halves][2 step parities], bar_saved[2 regions]
__host__ __device__ constexpr int off_tmem_ptr(bool exact) { return off_bars(exact) + kNumBars * 8; }
__host__ __device__ constexpr int smem_bytes(bool exact) { return off_tmem_ptr(exact) + 16; }
constexpr int kSmemBytes = smem_bytes(false);
static_assert(smem_bytes(true) <= 232448, "exact chain exceeds the 227 KB per-CTA shared memory limit");
static_assert(kMaxUnitBytes >= 256 * 128, "a hi or lo half-unit (<= 256 rows x 128 B) fills one ring slot");

enum : uint32_t { kFromOp = 1u, kWait0 = 2u, kWait1 = 4u, kFirst = 8u, kCommit0 = 16u, kPostWait1 = 64u, kOddRegion = 256u };
constexpr int total_units() {
  int n = 0;
  for (int s = 0; s < kBwdSteps; ++s) n += bwd_step_info(s).k_atoms;
  return n;
}
constexpr int kTileUnits = total_units();  // 28
struct ProgEntry { uint32_t x, y, z, w; };
struct ProgTable { ProgEntry e[32]; };
static_assert(kTileUnits <= 32, "program table too small");
constexpr uint32_t region_col_c(int s) { return (s & 1) ? 256u : 0u; }
// exact: w holds the unit's offset in stream_bwd_x3 (hi image; the lo image follows it), otherwise in the FP16 stream.
constexpr ProgTable make_prog(bool exact = false) {
  ProgTable t{};
  int i = 0;
  for (int s = 0; s < kBwdSteps; ++s) {
    const StepInfo si = bwd_step_info(s);
    const int nu = si.k_atoms;
    bool any_g2 = false;
    for (int j = 0; j < nu; ++j) any_g2 = any_g2 || bwd_unit_info(s, j).group == 2;
    for (int u = 0; u < nu; ++u, ++i) {
      const BwdUnit ui = bwd_unit_info(s, u);
      bool first_g1 = true, first_g2 = true;
      for (int j = 0; j < u; ++j) {
        if (bwd_unit_info(s, j).group == 1) first_g1 = false;
        if (bwd_unit_info(s, j).group == 2) first_g2 = false;
      }
      uint32_t flags = 0;
      if (ui.from_op) flags |= kFromOp;
      if (ui.group == 1 && first_g1) flags |= kWait0;
      if (ui.group == 2 && first_g2) flags |= kWait1;
      if (u == 0) flags |= kFirst;  // also: the step overwrites its region -> the savers must have read what lived there
      if (s & 1) flags |= kOddRegion;
      if (ui.last) flags |= kCommit0;
      if (u == nu - 1 && !any_g2) flags |= kPostWait1;
      const uint32_t d_col = region_col_c(s);
      const uint32_t a_col = (region_col_c(s) ^ 256u) + (uint32_t)(u - si.pe_first) * 64u;
      t.e[i].x = umma_idesc_f16(kTileM, ui.rows);
      t.e[i].y = d_col | (a_col << 16);
      t.e[i].z = flags;
      t.e[i].w = ((uint32_t)((exact ? 2 : 1) * bwd_unit_offset(s, u)) >> 4) | ((uint32_t)ui.rows << 20);
    }
  }
  return t;
}
__constant__ ProgTable c_prog = make_prog();
// The program a chain kernel runs: c_prog, or c_chain_prog_x3 (defined after the weight-gradient job table, so that table keeps its
// constant-bank offset).
template <bool EXACT> __device__ __forceinline__ const ProgTable& prog();

__device__ __forceinline__ uint32_t region_col(int s) { return (s & 1) ? 256u : 0u; }

// One 64-column slice of the accumulator: masked gradient -> FP16 (h a: columns [0,32), h b: [32,64)); EXACT: also the lo parts
// l a, l b (fp16(x - float(hi)), the split of the forward's epilogue).
template <bool EXACT>
__device__ __forceinline__ void bwd_epi_slice(uint32_t t_slice, uint2 m, uint32_t (&ha)[16], uint32_t (&hb)[16], uint32_t (&la)[16],
                                              uint32_t (&lb)[16]) {
  uint32_t va[32], vb[32];
  tmem_ld32(t_slice, va);
  tmem_ld32(t_slice + 32, vb);
  tmem_wait_ld();
#pragma unroll
  for (int j = 0; j < 32; j += 2) {
    const float a0 = ((m.x >> j) & 1u) ? __uint_as_float(va[j]) : 0.f;
    const float a1 = ((m.x >> (j + 1)) & 1u) ? __uint_as_float(va[j + 1]) : 0.f;
    const float b0 = ((m.y >> j) & 1u) ? __uint_as_float(vb[j]) : 0.f;
    const float b1 = ((m.y >> (j + 1)) & 1u) ? __uint_as_float(vb[j + 1]) : 0.f;
    ha[j / 2] = pack_f16x2(a0, a1);
    hb[j / 2] = pack_f16x2(b0, b1);
    if constexpr (EXACT) {
      const float2 ga = unpack_f16x2(ha[j / 2]), gb = unpack_f16x2(hb[j / 2]);
      la[j / 2] = pack_f16x2(a0 - ga.x, a1 - ga.y);
      lb[j / 2] = pack_f16x2(b0 - gb.x, b1 - gb.y);
    }
  }
}

// EXACT: the exact-gradient chain — hi/lo weight units, hi/lo d raw operand, every A operand as hi (+0) and lo (+32) of its slice,
// hi·W_hi + lo·W_hi + hi·W_lo per K slice as in the exact forward; the savers write the dY images of both record MiBs.
template <bool EXACT = false>
__global__ void __launch_bounds__(kThreads, 1) chain_kernel(const __grid_constant__ ChainParams p) {
  constexpr int NPART = EXACT ? 2 : 1;
  constexpr long long kRecStride = rec_stride(EXACT);
  constexpr int kBars = off_bars(EXACT), kTmemPtr = off_tmem_ptr(EXACT);
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t smem_base = smem_u32(smem);
  if ((smem_base & 1023u) != 0u) __trap();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const uint32_t bar_full = smem_base + kBars;
  const uint32_t bar_empty = bar_full + kNumSlots * 8;
  const uint32_t bar_aready = bar_empty + kNumSlots * 8;  // [2]
  const uint32_t bar_accfull = bar_aready + 16;           // [2] (only [0] used: one commit per step)
  const uint32_t bar_sv = bar_accfull + 16;               // [half][step & 1]: the step's FP16 output is in TMEM -> savers
  const uint32_t bar_saved = bar_sv + 32;                 // [region]: the savers have read the region -> MMA warp
  volatile uint32_t* tmem_ptr_s = reinterpret_cast<volatile uint32_t*>(smem + kTmemPtr);

  if (threadIdx.x == 0) {
    for (int i = 0; i < kNumSlots; ++i) {
      mbar_init(bar_full + i * 8, 1);
      mbar_init(bar_empty + i * 8, kCluster);
    }
    for (int h = 0; h < 2; ++h) {
      mbar_init(bar_aready + h * 8, kRowThreads / 32);
      mbar_init(bar_accfull + h * 8, 1);
      mbar_init(bar_sv + h * 16, kRowThreads / 32);
      mbar_init(bar_sv + h * 16 + 8, kRowThreads / 32);
      mbar_init(bar_saved + h * 8, 4);
    }
    mbar_fence_init();
  }
  if (warp == 1) {
    tmem_alloc(smem_base + kTmemPtr, 512);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < op_buffers(EXACT) * kTileM * 128 / 16; i += kThreads)  // operand chunks 1..7 of every row stay zero
    reinterpret_cast<uint4*>(smem + kOffOp)[i] = make_uint4(0u, 0u, 0u, 0u);
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr_s;
  const uint32_t cta_rank = cluster_ctarank();
  constexpr uint16_t kAllCtas = (1u << kCluster) - 1;

  const int first_in_cluster = (int)blockIdx.x - (int)cta_rank;
  const int n_iter = (p.n_units - first_in_cluster + (int)gridDim.x - 1) / (int)gridDim.x;
  const int tpu = p.tiles_c + p.tiles_f;
  const int n_tiles_cta = n_iter * tpu;

  if (warp == 0) {
    // ============================== weight producer ==============================
    reg_dec<kRegsLight>();
    uint32_t slot = 0, phase = 0, seq = 0;
    for (int j = 0; j < n_tiles_cta; ++j) {
      const int t = j % tpu;
      const uint8_t* base = p.wstream[t < p.tiles_c ? 0 : 1];
      for (int i = 0; i < kTileUnits; ++i) {
        const uint32_t w = prog<EXACT>().e[i].w;
        const uint32_t off = (w & 0xFFFFFu) << 4, bytes = (w >> 20) * 128u;
#pragma unroll
        for (int part = 0; part < NPART; ++part) {  // EXACT: the hi image, then the lo image that follows it in the stream
          mbar_wait(bar_empty + slot * 8, phase ^ 1);
          if (elect_one()) {
            mbar_arrive_expect_tx(bar_full + slot * 8, bytes);
            if ((seq % kCluster) == cta_rank)
              bulk_g2s_multicast(smem_base + kOffRing + slot * kMaxUnitBytes, base + off + part * bytes, bytes, bar_full + slot * 8, kAllCtas);
          }
          __syncwarp();
          ++seq;
          if (++slot == kNumSlots) { slot = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ============================== MMA issuer ==============================
    reg_dec<kRegsLight>();
    uint32_t slot = 0, phase = 0, ph_a0 = 0, ph_a1 = 0;
    uint32_t sv_pending = 0, sv_phase = 0;  // per region bit: a step's output lives there / parity of bar_saved
    const uint64_t op_desc = umma_smem_desc_sw128(smem_base + kOffOp);
    const uint64_t op_desc_lo = umma_smem_desc_sw128(smem_base + kOffOp + kTileM * 128);  // EXACT only
    for (int j = 0; j < n_tiles_cta; ++j) {
      for (int i = 0; i < kTileUnits; ++i) {
        const ProgEntry e = prog<EXACT>().e[i];
        if (e.z & kFirst) {  // first unit of a step
          const uint32_t rho = (e.z & kOddRegion) ? 1u : 0u;
          if (sv_pending & (1u << rho)) {
            mbar_wait(bar_saved + rho * 8, (sv_phase >> rho) & 1u);
            sv_phase ^= 1u << rho;
            tc_fence_after_sync();
          }
          sv_pending |= 1u << rho;
        }
        if (e.z & kWait0) {
          mbar_wait(bar_aready, ph_a0);
          ph_a0 ^= 1;
          tc_fence_after_sync();
        }
        if (e.z & kWait1) {
          mbar_wait(bar_aready + 8, ph_a1);
          ph_a1 ^= 1;
          tc_fence_after_sync();
        }
        const uint32_t d_tmem = tmem_base + (e.y & 0xFFFFu);
        const uint32_t a_tmem = tmem_base + (e.y >> 16);
        const uint32_t first = (e.z & kFirst) ? 0u : 1u;
#pragma unroll
        for (int part = 0; part < NPART; ++part) {  // EXACT: part 0 = W_hi (A hi and A lo), part 1 = W_lo (A hi)
          mbar_wait(bar_full + slot * 8, phase);
          tc_fence_after_sync();
          const uint64_t b_desc = umma_smem_desc_sw128(smem_base + kOffRing + slot * kMaxUnitBytes);
          if (elect_one()) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              const uint64_t bd = b_desc + (uint64_t)(ks * 2);
              const uint32_t acc_flag = (first | part | ks) ? 1u : 0u;
              if (e.z & kFromOp) {
                umma_ss(d_tmem, op_desc + (uint64_t)(ks * 2), bd, e.x, acc_flag);
                if (EXACT && part == 0) umma_ss(d_tmem, op_desc_lo + (uint64_t)(ks * 2), bd, e.x, 1);
              } else {
                umma_ts(d_tmem, a_tmem + ks * 8, bd, e.x, acc_flag);
                if (EXACT && part == 0) umma_ts(d_tmem, a_tmem + 32 + ks * 8, bd, e.x, 1);
              }
            }
            umma_commit_multicast(bar_empty + slot * 8, kAllCtas);
            if (part == NPART - 1 && (e.z & kCommit0)) umma_commit(bar_accfull);
          }
          __syncwarp();
          if (++slot == kNumSlots) { slot = 0; phase ^= 1; }
        }
        if (e.z & kPostWait1) {
          mbar_wait(bar_aready + 8, ph_a1);
          ph_a1 ^= 1;
        }
      }
    }
  } else if (warp >= 4 && warp < 12) {
    // ============================== row warps ==============================
    reg_inc<kRegsRow>();
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int ch = (warp - 4) >> 2;
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    uint32_t ph_acc = 0;
    const float scale = p.scal[0];

    // d raw of tile j -> FP16 operand row in shared memory (+ its transposed image for the weight-gradient kernel)
    auto write_operand = [&](int j) {
      const int unit = blockIdx.x + (j / tpu) * gridDim.x;
      const bool real = unit < p.n_units;
      const size_t gt = (size_t)unit * tpu + (j % tpu);
      if (ch == 0) {
        float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
        if (real) d = reinterpret_cast<const float4*>(p.draw)[gt * 128 + row];
        const uint32_t h01 = pack_f16x2(d.x * scale, d.y * scale), h23 = pack_f16x2(d.z * scale, d.w * scale);
        *reinterpret_cast<uint4*>(smem + kOffOp + row * 128 + ((0 ^ (row & 7)) << 4)) = make_uint4(h01, h23, 0u, 0u);
        uint32_t l01 = 0u, l23 = 0u;
        if constexpr (EXACT) {  // the scale is a power of two: d * scale is exact, its FP16 split as the epilogue's
          const float2 g01 = unpack_f16x2(h01), g23 = unpack_f16x2(h23);
          l01 = pack_f16x2(d.x * scale - g01.x, d.y * scale - g01.y);
          l23 = pack_f16x2(d.z * scale - g23.x, d.w * scale - g23.y);
          *reinterpret_cast<uint4*>(smem + kOffOp + kTileM * 128 + row * 128 + ((0 ^ (row & 7)) << 4)) = make_uint4(l01, l23, 0u, 0u);
        }
        if (real) {
          uint8_t* img = p.rec + gt * kRecStride + kRecDRaw + img_row_base(16, row);
          const uint32_t cr = (uint32_t)((row & 63) >> 3);
          *reinterpret_cast<uint16_t*>(img + 0 * 128 + ((cr ^ 0u) << 4)) = (uint16_t)(h01 & 0xFFFFu);
          *reinterpret_cast<uint16_t*>(img + 1 * 128 + ((cr ^ 1u) << 4)) = (uint16_t)(h01 >> 16);
          *reinterpret_cast<uint16_t*>(img + 2 * 128 + ((cr ^ 2u) << 4)) = (uint16_t)(h23 & 0xFFFFu);
          *reinterpret_cast<uint16_t*>(img + 3 * 128 + ((cr ^ 3u) << 4)) = (uint16_t)(h23 >> 16);
          if constexpr (EXACT) {
            *reinterpret_cast<uint16_t*>(img + kRecLo + 0 * 128 + ((cr ^ 0u) << 4)) = (uint16_t)(l01 & 0xFFFFu);
            *reinterpret_cast<uint16_t*>(img + kRecLo + 1 * 128 + ((cr ^ 1u) << 4)) = (uint16_t)(l01 >> 16);
            *reinterpret_cast<uint16_t*>(img + kRecLo + 2 * 128 + ((cr ^ 2u) << 4)) = (uint16_t)(l23 & 0xFFFFu);
            *reinterpret_cast<uint16_t*>(img + kRecLo + 3 * 128 + ((cr ^ 3u) << 4)) = (uint16_t)(l23 >> 16);
          }
        }
      } else if (real) {  // rows 4..15 of the image are zero
        uint8_t* img = p.rec + gt * kRecStride + kRecDRaw + img_row_base(16, row);
        const uint32_t cr = (uint32_t)((row & 63) >> 3);
#pragma unroll
        for (int part = 0; part < NPART; ++part) {
#pragma unroll
          for (int k = 4; k < 16; ++k) *reinterpret_cast<uint16_t*>(img + part * kRecLo + k * 128 + ((cr ^ (uint32_t)(k & 7)) << 4)) = 0;
        }
      }
      fence_proxy_async_smem();
    };

    if (n_tiles_cta > 0) write_operand(0);
    for (int j = 0; j < n_tiles_cta; ++j) {
      const int unit = blockIdx.x + (j / tpu) * gridDim.x;
      const bool real = unit < p.n_units;
      uint8_t* rec = real ? p.rec + ((size_t)unit * tpu + (j % tpu)) * kRecStride : nullptr;
      const uint32_t* masks = reinterpret_cast<const uint32_t*>(rec + kRecMask);
      __syncwarp();
      if (lane == 0) {  // operand of tile j is in place: both gates of step 0
        mbar_arrive(bar_aready);
        mbar_arrive(bar_aready + 8);
      }
      for (int s = 0; s < kBwdSteps; ++s) {
        const int L = 8 - s;  // forward layer whose pre-activation gradient this step produces
        const bool two = s >= 3;
        const uint32_t t_acc = t_lane + region_col(s);
        const int W = rec_width(L);
        uint2 m0 = make_uint2(0u, 0u), m1 = make_uint2(0u, 0u);
        if (real) {
          m0 = *reinterpret_cast<const uint2*>(masks + (L * 128 + row) * 8 + 2 * ch);
          if (two) m1 = *reinterpret_cast<const uint2*>(masks + (L * 128 + row) * 8 + 4 + 2 * ch);
        }
        mbar_wait(bar_accfull, ph_acc);
        ph_acc ^= 1;
        tc_fence_after_sync();
        const uint32_t par = (uint32_t)(s & 1);
        {  // half 0: output columns [64 ch, 64 ch + 64).  The FP16 result goes back to TMEM in place: A operand of the next step
           // and (every step, also the last) what the saver warps write to the record.
          const int c0 = 64 * ch;
          uint32_t ha[16], hb[16], la[16], lb[16];
          bwd_epi_slice<EXACT>(t_acc + c0, m0, ha, hb, la, lb);
          tmem_st16(t_acc + c0, ha);
          tmem_st16(t_acc + c0 + 16, hb);
          if constexpr (EXACT) {
            tmem_st16(t_acc + c0 + 32, la);
            tmem_st16(t_acc + c0 + 48, lb);
          }
          tmem_wait_st();
          tc_fence_before_sync();
          __syncwarp();
          if (lane == 0) {
            if (s < kBwdSteps - 1) mbar_arrive(bar_aready);
            mbar_arrive(bar_sv + par * 8);
          }
        }
        if (two) {  // half 1: columns [128 + 64 ch, ...)
          const int c0 = 128 + 64 * ch;
          uint32_t ha[16], hb[16], la[16], lb[16];
          bwd_epi_slice<EXACT>(t_acc + c0, m1, ha, hb, la, lb);
          tmem_st16(t_acc + c0, ha);
          tmem_st16(t_acc + c0 + 16, hb);
          if constexpr (EXACT) {
            tmem_st16(t_acc + c0 + 32, la);
            tmem_st16(t_acc + c0 + 48, lb);
          }
          tmem_wait_st();
          tc_fence_before_sync();
          __syncwarp();
          if (lane == 0) {
            if (s < kBwdSteps - 1) mbar_arrive(bar_aready + 8);
            mbar_arrive(bar_sv + 16 + par * 8);
          }
        } else if (s < kBwdSteps - 1) {
          tc_fence_before_sync();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_aready + 8);
        }
        if (s == 3 && j + 1 < n_tiles_cta) write_operand(j + 1);  // steps 0 and 3 of tile j no longer read the operand
      }
    }
    tc_fence_before_sync();
  } else if (warp >= 12) {
    // ============================== record savers ==============================
    // bar_sv[half][s & 1] cannot run more than one phase ahead of this warp: the step that next completes the same barrier is
    // s + 2 (or a step of the next tile in the same region), whose MMAs wait for bar_saved of step s.
    reg_dec<kRegsSaver>();
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    uint32_t sv_ph = 0;  // bit (half * 2 + parity): phase of bar_sv[half][parity]
    for (int j = 0; j < n_tiles_cta; ++j) {
      const int unit = blockIdx.x + (j / tpu) * gridDim.x;
      uint8_t* rec = unit < p.n_units ? p.rec + ((size_t)unit * tpu + (j % tpu)) * kRecStride : nullptr;
#pragma unroll 1
      for (int s = 0; s < kBwdSteps; ++s) {
        const int L = 8 - s, W = rec_width(L);
        const uint32_t par = (uint32_t)(s & 1);
        const uint32_t t_reg = t_lane + region_col(s);
        uint8_t* img = rec ? rec + rec_dy_off(L) + img_row_base(W, row) : nullptr;
        const int n_slices = W >> 6;
#pragma unroll 1
        for (int i = 0; i < n_slices; ++i) {
          if ((i & 1) == 0) {
            const int h = i >> 1;
            const uint32_t bit = 1u << (h * 2 + par);
            mbar_wait(bar_sv + h * 16 + par * 8, (sv_ph & bit) ? 1u : 0u);
            sv_ph ^= bit;
            tc_fence_after_sync();
          }
          // EXACT: two passes per slice (hi columns, then lo columns at +32), so the savers stay at 80 registers
#pragma unroll
          for (int part = 0; part < NPART; ++part) {
            uint32_t v[32];
            tmem_ld32(t_reg + 64 * i + 32 * part, v);
            tmem_wait_ld();
            if (i == n_slices - 1 && part == NPART - 1) {  // the whole region has been read
              tc_fence_before_sync();
              __syncwarp();
              if (lane == 0) mbar_arrive(bar_saved + par * 8);
            }
            if (img) {
              uint8_t* dst = img + part * kRecLo;
              uint32_t h0[16], h1[16];
#pragma unroll
              for (int k = 0; k < 16; ++k) { h0[k] = v[k]; h1[k] = v[16 + k]; }
              store_t32(dst, row, 64 * i, h0);
              store_t32(dst, row, 64 * i + 32, h1);
            }
          }
        }
      }
    }
    tc_fence_before_sync();
  } else {
    reg_dec<kRegsLight>();  // warps 2, 3: idle, but setmaxnreg is a warpgroup-wide instruction
  }

  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace chain

// ================================================================================================
// 3. weight-gradient kernel
// ================================================================================================
namespace dw {

constexpr int kThreads = 192;  // warp 0 producer, warp 1 MMA issuer, warps 2..5 epilogue (one per TMEM lane quadrant)
constexpr int kStages = 4;
constexpr int kStageBytes = 16384 + 32768;       // one r-atom (64 sample rows): A [128 features x 128 B], B [<=256 features x 128 B]
// EXACT (exact-gradient records): a stage holds the hi images as above and the lo images (second record MiB) kStageBytes after
// them, so 2 stages of 96 KB take the space of 4 x 48 KB.
__host__ __device__ constexpr int stages(bool exact) { return exact ? 2 : kStages; }
__host__ __device__ constexpr int stage_bytes(bool exact) { return exact ? 2 * kStageBytes : kStageBytes; }
__host__ __device__ constexpr int stage_a_off(int part) { return part * kStageBytes; }           // part 0 = hi, 1 = lo
__host__ __device__ constexpr int stage_b_off(int part) { return part * kStageBytes + 16384; }
// bytes one stage (one r-atom of one tile) brings in for a job whose B image has b_rows features
__host__ __device__ constexpr uint32_t stage_tx(bool exact, int b_rows) { return (exact ? 2u : 1u) * (16384u + (uint32_t)b_rows * 128u); }
static_assert(stages(true) * stage_bytes(true) == kStages * kStageBytes, "both variants share the shared-memory map");
constexpr int kOffOnes = kStages * kStageBytes;  // [16 rows x 64 r]: row 0 = 1.0 (bias = column sums of dY)
constexpr int kOffBars = kOffOnes + 2048;
constexpr int kOffTmemPtr = kOffBars + (2 * kStages + 2) * 8;
constexpr int kSmemBytes = kOffTmemPtr + 16;
constexpr uint32_t kBiasCol = 256;

struct Job {
  int a_off, a_rows, a_half;  // A image (M side): record offset, features in the image, which 128-feature half
  int b_off, b_rows;          // B image (N side): record offset, features (= MMA N)
  int bias_layer;             // >= 0: also accumulate column sums of A into the bias of this layer
  int out_off, out_ld, out_row0;
};
// Jobs are dealt to kGroups groups of CTAs; within a group every CTA runs the group's jobs over its own share of the tiles (fewer
// accumulator drains and atomics than every CTA running every job).  The kernel is HBM-bound (each job streams its two images of
// every tile once), so the groups are balanced by BYTES per tile (172..200 KB each), and groups 2q / 2q+1 are the two
// 128-feature output halves of the SAME layers in the SAME order: they run on neighbouring CTAs over the same tiles at the same
// time, so the B image both need (the layer's whole input, 2/3 of a job's bytes) comes from HBM once and from L2 the second time.
constexpr int kNumJobs = 21;
constexpr int kGroups = 8;
struct JobTable { Job j[kNumJobs]; int group_begin[kGroups + 1]; };
constexpr Job half_job(int dy_layer, int h, int b_off, int b_rows, int bias_layer, int out_off) {
  return Job{rec_dy_off(dy_layer), 256, h, b_off, b_rows, bias_layer, out_off, b_rows, 128 * h};
}
constexpr JobTable make_jobs() {
  JobTable t{};
  int i = 0, g = 0;
  for (int h = 0; h < 2; ++h) {  // groups 0, 1: layers_xyz.1, .2
    t.group_begin[g++] = i;
    t.j[i++] = half_job(1, h, rec_x_off(0), 256, 1, kAcc1);
    t.j[i++] = half_job(2, h, rec_x_off(1), 256, 2, kAcc2);
  }
  for (int h = 0; h < 2; ++h) {  // groups 2, 3: layers_xyz.4, .5
    t.group_begin[g++] = i;
    t.j[i++] = half_job(4, h, rec_x_off(3), 256, 4, kAcc4);
    t.j[i++] = half_job(5, h, rec_x_off(4), 256, 5, kAcc5);
  }
  for (int h = 0; h < 2; ++h) {  // groups 4, 5: the skip layer (hidden part, then its PE part) and layers_xyz.0 (dY0 x PE)
    t.group_begin[g++] = i;
    t.j[i++] = half_job(3, h, rec_x_off(2), 256, -1, kAcc3b);
    t.j[i++] = half_job(3, h, kRecPE, 64, 3, kAcc3a);
    t.j[i++] = half_job(0, h, kRecPE, 64, 0, kAcc0);
  }
  t.group_begin[g++] = i;          // group 6: everything that reads dY6 or h5
  t.j[i++] = Job{rec_dy_off(6), 128, 0, rec_x_off(5), 256, 6, kAcc6, 256, 0};     // d M1
  t.j[i++] = Job{rec_dy_off(6), 128, 0, kRecPEd, 32, -1, kAcc6d, 32, 0};          // d layers_dir.0[:, 256:280]
  t.j[i++] = Job{rec_x_off(5), 256, 0, kRecDRaw, 16, -1, kAccSig, 16, 0};         // h5^T . d raw, first half
  t.group_begin[g++] = i;          // group 7: its second half and the rest of the direction branch
  t.j[i++] = Job{rec_x_off(5), 256, 1, kRecDRaw, 16, -1, kAccSig, 16, 128};
  t.j[i++] = Job{rec_dy_off(7), 128, 0, rec_x_off(6), 128, 7, kAcc7, 128, 0};
  t.j[i++] = Job{rec_dy_off(8), 128, 0, rec_x_off(7), 128, 8, kAcc8, 128, 0};
  t.j[i++] = Job{rec_x_off(8), 128, 0, kRecDRaw, 16, -1, kAcc9, 16, 0};           // g2^T . d raw
  t.group_begin[g] = i;
  return t;
}
static_assert(make_jobs().group_begin[kGroups] == kNumJobs, "job table");
__constant__ JobTable c_jobs = make_jobs();

}  // namespace dw

__constant__ chain::ProgTable c_chain_prog_x3 = chain::make_prog(true);
namespace chain {
template <> __device__ __forceinline__ const ProgTable& prog<false>() { return c_prog; }
template <> __device__ __forceinline__ const ProgTable& prog<true>() { return c_chain_prog_x3; }
}  // namespace chain

namespace dw {

// EXACT: exact-gradient records — per ks A_hi·B_hi + A_hi·B_lo + A_lo·B_hi, and A_hi·1 + A_lo·1 for the bias column.
template <bool EXACT = false>
__global__ void __launch_bounds__(kThreads, 1) dw_kernel(const __grid_constant__ DwParams p) {
  constexpr int NSTAGE = stages(EXACT), NPART = EXACT ? 2 : 1;
  constexpr int kStride = stage_bytes(EXACT);
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t smem_base = smem_u32(smem);
  if ((smem_base & 1023u) != 0u) __trap();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // this CTA: network x job group (blockIdx.x % kGroups) x a contiguous share of the network's tiles
  const int group = (int)blockIdx.x % kGroups;
  int part = (int)blockIdx.x / kGroups;
  const int net = (part >= p.parts[0]) ? 1 : 0;
  if (net) part -= p.parts[0];
  const int parts = p.parts[net];
  const int t_cnt = p.t_cnt[net], t_base = p.t_base[net];
  const int total = p.n_units * t_cnt;
  const int per = (total + parts - 1) / parts;
  const int j0 = part * per;
  const int j1 = min(total, j0 + per);
  if (part >= parts || j0 >= j1) return;  // uniform for the whole CTA
  const int job0 = c_jobs.group_begin[group], job1 = c_jobs.group_begin[group + 1];

  const uint32_t bar_full = smem_base + kOffBars;      // [NSTAGE]
  const uint32_t bar_empty = bar_full + NSTAGE * 8;    // [NSTAGE]
  const uint32_t bar_accfull = bar_empty + NSTAGE * 8;
  const uint32_t bar_accempty = bar_accfull + 8;
  volatile uint32_t* tmem_ptr_s = reinterpret_cast<volatile uint32_t*>(smem + kOffTmemPtr);

  if (threadIdx.x == 0) {
    for (int i = 0; i < NSTAGE; ++i) {
      mbar_init(bar_full + i * 8, 1);
      mbar_init(bar_empty + i * 8, 1);
    }
    mbar_init(bar_accfull, 1);
    mbar_init(bar_accempty, 4);
    mbar_fence_init();
  }
  if (warp == 1) {
    tmem_alloc(smem_base + kOffTmemPtr, 512);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < 2048 / 4; i += kThreads)  // row 0 (first 128 bytes) = FP16 ones, rows 1..15 = 0
    reinterpret_cast<uint32_t*>(smem + kOffOnes)[i] = (i < 32) ? 0x3C003C00u : 0u;
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr_s;

  auto tile_rec = [&](int j) -> const uint8_t* {
    const int u = j / t_cnt, t = j - u * t_cnt;
    return p.rec + ((size_t)u * p.tpu + t_base + t) * rec_stride(EXACT);
  };

  if (warp == 0) {
    // ============================== producer ==============================
    uint32_t stage = 0, phase = 0;
    for (int job = job0; job < job1; ++job) {
      const Job J = c_jobs.j[job];
      const uint32_t b_bytes = (uint32_t)J.b_rows * 128u;
      for (int j = j0; j < j1; ++j) {
        const uint8_t* rec = tile_rec(j);
        for (int a = 0; a < 2; ++a) {
          mbar_wait(bar_empty + stage * 8, phase ^ 1);
          if (elect_one()) {
            const uint32_t st0 = smem_base + stage * kStride;
            mbar_arrive_expect_tx(bar_full + stage * 8, stage_tx(EXACT, J.b_rows));
#pragma unroll
            for (int part = 0; part < NPART; ++part) {  // EXACT: the hi images, then the lo images of the second record MiB
              const uint8_t* r = rec + part * kRecLo;
              bulk_g2s(st0 + stage_a_off(part), r + J.a_off + a * J.a_rows * 128 + J.a_half * 16384, 16384, bar_full + stage * 8);
              bulk_g2s(st0 + stage_b_off(part), r + J.b_off + a * J.b_rows * 128, b_bytes, bar_full + stage * 8);
            }
          }
          __syncwarp();
          if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ============================== MMA issuer ==============================
    uint32_t stage = 0, phase = 0, acc_phase = 0;
    const uint64_t ones_desc = umma_smem_desc_sw128(smem_base + kOffOnes);
    const uint32_t idesc_bias = umma_idesc_f16(128, 16);
    for (int job = job0; job < job1; ++job) {
      const Job J = c_jobs.j[job];
      const uint32_t idesc = umma_idesc_f16(128, J.b_rows);
      mbar_wait(bar_accempty, acc_phase ^ 1);  // the epilogue has drained the previous job's accumulator
      tc_fence_after_sync();
      for (int j = j0; j < j1; ++j) {
        for (int a = 0; a < 2; ++a) {
          mbar_wait(bar_full + stage * 8, phase);
          tc_fence_after_sync();
          const uint32_t sa = smem_base + stage * kStride + stage_a_off(0), sb = smem_base + stage * kStride + stage_b_off(0);
          if (elect_one()) {
            const uint64_t ad = umma_smem_desc_sw128(sa), bd = umma_smem_desc_sw128(sb);
            const uint32_t sal = smem_base + stage * kStride + stage_a_off(1), sbl = smem_base + stage * kStride + stage_b_off(1);
            const uint64_t adl = umma_smem_desc_sw128(sal), bdl = umma_smem_desc_sw128(sbl);  // EXACT only
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              const uint32_t accf = ((j - j0) | a | ks) ? 1u : 0u;
              umma_ss(tmem_base, ad + (uint64_t)(ks * 2), bd + (uint64_t)(ks * 2), idesc, accf);
              if constexpr (EXACT) {
                umma_ss(tmem_base, ad + (uint64_t)(ks * 2), bdl + (uint64_t)(ks * 2), idesc, 1u);
                umma_ss(tmem_base, adl + (uint64_t)(ks * 2), bd + (uint64_t)(ks * 2), idesc, 1u);
              }
              if (J.bias_layer >= 0) {
                umma_ss(tmem_base + kBiasCol, ad + (uint64_t)(ks * 2), ones_desc + (uint64_t)(ks * 2), idesc_bias, accf);
                if (EXACT) umma_ss(tmem_base + kBiasCol, adl + (uint64_t)(ks * 2), ones_desc + (uint64_t)(ks * 2), idesc_bias, 1u);
              }
            }
            umma_commit(bar_empty + stage * 8);
            if (j == j1 - 1 && a == 1) umma_commit(bar_accfull);
          }
          __syncwarp();
          if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
        }
      }
      acc_phase ^= 1;
    }
  } else {
    // ============================== epilogue ==============================
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    const float inv = p.scal[1];
    uint32_t acc_phase = 0;
    for (int job = job0; job < job1; ++job) {
      const Job J = c_jobs.j[job];
      mbar_wait(bar_accfull, acc_phase);
      acc_phase ^= 1;
      tc_fence_after_sync();
      float* out = p.acc[net] + J.out_off + (size_t)(J.out_row0 + row) * J.out_ld;
      if (J.b_rows == 16) {
        uint32_t v[16];
        tmem_ld16(t_lane, v);
        tmem_wait_ld();
#pragma unroll
        for (int c = 0; c < 16; ++c) atomicAdd(out + c, __uint_as_float(v[c]) * inv);
      } else {
        for (int c0 = 0; c0 < J.b_rows; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(t_lane + c0, v);
          tmem_wait_ld();
#pragma unroll
          for (int c = 0; c < 32; ++c) atomicAdd(out + c0 + c, __uint_as_float(v[c]) * inv);
        }
      }
      if (J.bias_layer >= 0) {
        uint32_t v[4];
        tmem_ld4(t_lane + kBiasCol, v);
        tmem_wait_ld();
        atomicAdd(p.acc[net] + acc_bias_off(J.bias_layer) + J.out_row0 + row, __uint_as_float(v[0]) * inv);
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_accempty);
    }
  }

  __syncthreads();
  if (warp == 1) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace dw

// ================================================================================================
// 4. finalize: accumulators (folded parametrisation) -> reference parameter gradients
// ================================================================================================
struct FinArgs {
  const float* p[26];  // FP32 master parameters (device)
  float* g[26];        // gradient outputs (device; layers_dir.3.* may be null)
  const float* acc;    // this network's accumulators
  const float* cond;   // [108] = [expression / 3 ; latent]
};
__device__ __forceinline__ int fin_numel(int t) {
  switch (t) {
    case 0: return 256 * 171;
    case 6: return 256 * 427;
    case 2: case 4: case 8: case 10: case 12: return 65536;
    case 1: case 3: case 5: case 7: case 9: case 11: case 13: case 14: return 256;
    case 15: return 1;
    case 16: return 128 * 280;
    case 18: case 20: return 128 * 128;
    case 17: case 19: case 21: return 128;
    case 24: return 3 * 128;
    case 25: return 3;
    default: return 0;  // layers_dir.3.*: unused by the forward (models.py:257) -> no gradient
  }
}
// ONE launch finishes both networks: blockIdx.y = network; blockIdx.x walks the 26 tensors back to back in 256-element blocks
// (2.2 k blocks per network instead of a 427 x 26 grid that is mostly empty); the last block of network 0 computes d latent.
struct FinAll { FinArgs net[2]; int nets; float* latent_out; };
__device__ __forceinline__ int fin_blocks(int t) { return (fin_numel(t) + 255) >> 8; }
__device__ void latent_grad_block(const FinAll& f);
__global__ void __launch_bounds__(256) finalize_kernel(const FinAll f) {
  const FinArgs& a = f.net[blockIdx.y];
  int b = blockIdx.x, t = 0;
  while (t < 26 && b >= fin_blocks(t)) { b -= fin_blocks(t); ++t; }
  if (t == 26) {  // the block after the last tensor
    if (blockIdx.y == 0 && b == 0 && f.latent_out) latent_grad_block(f);
    return;
  }
  const int e = b * 256 + threadIdx.x;
  if (e >= fin_numel(t) || a.g[t] == nullptr) return;
  const float* acc = a.acc;
  const float* b6 = acc + acc_bias_off(6);
  const float dbs = acc[kAccBRaw + 3];  // d (fc_alpha.bias + wa . bf)
  float v = 0.f;
  switch (t) {
    case 0: {
      const int n = e / 171, k = e - n * 171;
      v = (k < kDimXyz) ? acc[kAcc0 + n * 64 + k] : acc[acc_bias_off(0) + n] * a.cond[k - kDimXyz];
      break;
    }
    case 6: {
      const int n = e / 427, k = e - n * 427;
      v = (k < kDimXyz) ? acc[kAcc3a + n * 64 + k]
          : (k < kDimXyz + kDimCond) ? acc[acc_bias_off(3) + n] * a.cond[k - kDimXyz]
                                     : acc[kAcc3b + n * 256 + (k - kDimXyz - kDimCond)];
      break;
    }
    case 1: v = acc[acc_bias_off(0) + e]; break;
    case 2: v = acc[kAcc1 + e]; break;
    case 3: v = acc[acc_bias_off(1) + e]; break;
    case 4: v = acc[kAcc2 + e]; break;
    case 5: v = acc[acc_bias_off(2) + e]; break;
    case 7: v = acc[acc_bias_off(3) + e]; break;
    case 8: v = acc[kAcc4 + e]; break;
    case 9: v = acc[acc_bias_off(4) + e]; break;
    case 10: v = acc[kAcc5 + e]; break;
    case 11: v = acc[acc_bias_off(5) + e]; break;
    case 12: {  // fc_feat.weight[j][k] = sum_i Wd0[i][j] dM1[i][k] + wa[j] dm2[k]
      const int j = e >> 8, k = e & 255;
      float s = a.p[14][j] * acc[kAccSig + k * 16 + 3];
      for (int i = 0; i < 128; ++i) s = fmaf(a.p[16][i * 280 + j], acc[kAcc6 + i * 256 + k], s);
      v = s;
      break;
    }
    case 13: {  // fc_feat.bias[j] = sum_i Wd0[i][j] db6[i] + wa[j] dbs
      float s = a.p[14][e] * dbs;
      for (int i = 0; i < 128; ++i) s = fmaf(a.p[16][i * 280 + e], b6[i], s);
      v = s;
      break;
    }
    case 14: return;  // fc_alpha.weight: 256 dot products of length 256 -> fin_dir0_kernel (one warp each, coalesced)
    case 15: v = dbs; break;
    case 16: {  // layers_dir.0.weight[i][j]: j < 256: sum_k dM1[i][k] Wf[j][k] + db6[i] bf[j]; else direction columns
      const int i = e / 280, j = e - i * 280;
      if (j < 256) return;  // written by fin_dir0_kernel (one warp per element, coalesced along k)
      v = acc[kAcc6d + i * 32 + (j - 256)];
      break;
    }
    case 17: v = b6[e]; break;
    case 18: v = acc[kAcc7 + e]; break;
    case 19: v = acc[acc_bias_off(7) + e]; break;
    case 20: v = acc[kAcc8 + e]; break;
    case 21: v = acc[acc_bias_off(8) + e]; break;
    case 24: { const int n = e >> 7, k = e & 127; v = acc[kAcc9 + k * 16 + n]; break; }
    case 25: v = acc[kAccBRaw + e]; break;
    default: break;
  }
  a.g[t][e] = v;
}

// layers_dir.0.weight[i][j], j < 256:  sum_k dM1[i][k] Wf[j][k] + db6[i] bf[j].  One warp per output element, lanes along k.
__global__ void fin_dir0_kernel(const FinAll f) {
  const FinArgs& a = f.net[blockIdx.y];
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (w >= 128 * 256) {  // fc_alpha.weight[0][j] = sum_k dm2[k] Wf[j][k] + dbs bf[j]
    const int j = w - 128 * 256;
    if (j >= 256 || a.g[14] == nullptr) return;
    const float* wf = a.p[12] + j * 256;
    float s = 0.f;
#pragma unroll
    for (int k = lane; k < 256; k += 32) s = fmaf(a.acc[kAccSig + k * 16 + 3], wf[k], s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) a.g[14][j] = s + a.acc[kAccBRaw + 3] * a.p[13][j];
    return;
  }
  const int i = w >> 8, j = w & 255;
  const float* dm1 = a.acc + kAcc6 + i * 256;
  const float* wf = a.p[12] + j * 256;
  float s = 0.f;
#pragma unroll
  for (int k = lane; k < 256; k += 32) s = fmaf(dm1[k], wf[k], s);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) a.g[16][i * 280 + j] = s + a.acc[acc_bias_off(6) + i] * a.p[13][j];
}

// d latent[j] = sum over networks, n of W0[n][139 + j] db0[n] + W3[n][139 + j] db3[n]
__device__ void latent_grad_block(const FinAll& f) {  // one block of 256 threads: thread = (n-chunk of 32 rows, j)
  __shared__ float part[8][kDimLatent];
  const int j = threadIdx.x & 31, c = threadIdx.x >> 5;
  float s = 0.f;
  for (int net = 0; net < f.nets; ++net) {
    const float* b0 = f.net[net].acc + acc_bias_off(0);
    const float* b3 = f.net[net].acc + acc_bias_off(3);
    const float* w0 = f.net[net].p[0];
    const float* w3 = f.net[net].p[6];
    for (int n = c * 32; n < c * 32 + 32; ++n) {
      s = fmaf(w0[n * 171 + kDimXyz + kDimExpr + j], b0[n], s);
      s = fmaf(w3[(size_t)n * 427 + kDimXyz + kDimExpr + j], b3[n], s);
    }
  }
  part[c][j] = s;
  __syncthreads();
  if (c == 0) {
    float t = 0.f;
    for (int k = 0; k < 8; ++k) t += part[k][j];
    f.latent_out[j] = t;
  }
}

// ================================================================================================
// host-side launchers
// ================================================================================================
int debug_prog_chain(int index, uint32_t* out) {
  constexpr chain::ProgTable t = chain::make_prog();
  if (index < 0) return chain::kTileUnits;
  if (index >= chain::kTileUnits) return -1;
  out[0] = t.e[index].x; out[1] = t.e[index].y; out[2] = t.e[index].z; out[3] = t.e[index].w;
  return 4;
}
int debug_jobs_dw(int index, uint32_t* out) {
  constexpr dw::JobTable t = dw::make_jobs();
  if (index < 0) return dw::kNumJobs;
  if (index >= dw::kNumJobs) return -1;
  const dw::Job& j = t.j[index];
  const int v[9] = {j.a_off, j.a_rows, j.a_half, j.b_off, j.b_rows, j.bias_layer, j.out_off, j.out_ld, j.out_row0};
  for (int i = 0; i < 9; ++i) out[i] = (uint32_t)v[i];
  int g = 0;
  while (g + 1 < dw::kGroups && t.group_begin[g + 1] <= index) ++g;
  out[9] = (uint32_t)g;
  return 10;
}

// Exact-gradient chain program, one entry per LOAD (two per unit: hi, lo): the unit's program entry with w = this part's offset in
// stream_bwd_x3, then part, the A operand's lo TMEM column (0xFFFFFFFF: from the shared-memory operand), the kernel's shared-memory
// bytes, ring slot bytes, ring slots, d raw operand buffers.
int debug_prog_chain_exact(int index, uint32_t* out) {
  constexpr chain::ProgTable t = chain::make_prog(true);
  if (index < 0) return 2 * chain::kTileUnits;
  if (index >= 2 * chain::kTileUnits) return -1;
  const chain::ProgEntry& e = t.e[index / 2];
  const uint32_t part = (uint32_t)(index & 1), bytes = (e.w >> 20) * 128u;
  out[0] = e.x; out[1] = e.y; out[2] = e.z;
  out[3] = ((((e.w & 0xFFFFFu) << 4) + part * bytes) >> 4) | (e.w & ~0xFFFFFu);
  out[4] = part;
  out[5] = (e.z & chain::kFromOp) ? 0xFFFFFFFFu : (e.y >> 16) + 32u;
  out[6] = (uint32_t)chain::smem_bytes(true); out[7] = (uint32_t)kMaxUnitBytes; out[8] = (uint32_t)chain::kNumSlots;
  out[9] = (uint32_t)chain::op_buffers(true);
  return 10;
}
// Exact-gradient weight-gradient stage layout, one entry per job: shared-memory offsets inside a stage of A hi, B hi, A lo, B lo,
// stage bytes, stages, bytes the job loads per tile (two r-atoms), the same for the FP16 kernel, the kernel's shared-memory bytes,
// record offset of the lo MiB.
int debug_stages_dw_exact(int index, uint32_t* out) {
  constexpr dw::JobTable t = dw::make_jobs();
  if (index < 0) return dw::kNumJobs;
  if (index >= dw::kNumJobs) return -1;
  const int b_rows = t.j[index].b_rows;
  out[0] = dw::stage_a_off(0); out[1] = dw::stage_b_off(0); out[2] = dw::stage_a_off(1); out[3] = dw::stage_b_off(1);
  out[4] = (uint32_t)dw::stage_bytes(true); out[5] = (uint32_t)dw::stages(true);
  out[6] = 2u * dw::stage_tx(true, b_rows); out[7] = 2u * dw::stage_tx(false, b_rows);
  out[8] = (uint32_t)dw::kSmemBytes; out[9] = (uint32_t)kRecLo;
  return 10;
}

cudaError_t train_kernels_setup() {
  cudaError_t e = cudaFuncSetAttribute(chain::chain_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, chain::kSmemBytes);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(chain::chain_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, chain::smem_bytes(true));
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(dw::dw_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, dw::kSmemBytes);
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(dw::dw_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, dw::kSmemBytes);
}

cudaError_t launch_composite_bwd(const CompBwdParams& q, float* scal, cudaStream_t st, long long* launches) {
  const int n = (q.nf > 0 ? 2 : 1) * q.n_rays;
  composite_bwd_kernel<<<(n + 7) / 8, 256, 0, st>>>(q);  // one warp per (ray, pass)
  ++*launches;
  scale_kernel<<<1, 1, 0, st>>>(q.absmax, scal);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_chain(const ChainParams& p, bool exact_grad, int num_sms, cudaStream_t st, long long* launches) {
  int grid = p.n_units < num_sms ? p.n_units : num_sms;
  if (grid <= 0) return cudaSuccess;
  grid = (grid + chain::kCluster - 1) / chain::kCluster * chain::kCluster;
  if (grid > num_sms) grid = num_sms / chain::kCluster * chain::kCluster;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(chain::kThreads);
  cfg.dynamicSmemBytes = exact_grad ? chain::smem_bytes(true) : chain::kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = chain::kCluster;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = exact_grad ? cudaLaunchKernelEx(&cfg, chain::chain_kernel<true>, p) : cudaLaunchKernelEx(&cfg, chain::chain_kernel<false>, p);
  ++*launches;
  return e != cudaSuccess ? e : cudaGetLastError();
}

// CTAs per job group for the two networks: `num_sms / kGroups` parts split in proportion to the networks' tile counts
// (64c + 64f: 1 : 2 -> 6 + 12 on 148 SMs, 171 tiles per CTA either way), at least one part per non-empty network, never more
// parts than tiles.  Host logic, exposed to the tests through nfb_debug_schedule(4, ...).
void dw_split(int num_sms, long long tot0, long long tot1, int* parts0, int* parts1) {
  int parts = num_sms / dw::kGroups;
  if (parts < 1) parts = 1;
  if (tot0 > 0 && tot1 > 0 && parts < 2) parts = 2;  // CTAs are independent: more CTAs than SMs only serialises them
  int p0 = tot1 <= 0 ? (tot0 > 0 ? parts : 0) : (tot0 <= 0 ? 0 : (int)((parts * tot0 + (tot0 + tot1) / 2) / (tot0 + tot1)));
  if (tot0 > 0 && p0 < 1) p0 = 1;
  if (tot1 > 0 && p0 > parts - 1) p0 = parts - 1;
  int p1 = tot1 > 0 ? parts - p0 : 0;
  if (p0 > tot0) p0 = (int)tot0;
  if (p1 > tot1) p1 = (int)tot1;
  *parts0 = p0;
  *parts1 = p1;
}
int debug_dw_split(uint32_t* io) {  // in: num_sms, tiles of network 0, tiles of network 1; out: parts0, parts1, groups
  int p0 = 0, p1 = 0;
  dw_split((int)io[0], (long long)io[1], (long long)io[2], &p0, &p1);
  io[0] = (uint32_t)p0; io[1] = (uint32_t)p1; io[2] = (uint32_t)dw::kGroups;
  return 3;
}

cudaError_t launch_dw(const DwParams& p_in, bool exact_grad, int num_sms, cudaStream_t st, long long* launches) {
  DwParams p = p_in;
  const long long tot0 = (long long)p.n_units * p.t_cnt[0], tot1 = (long long)p.n_units * p.t_cnt[1];
  if (tot0 + tot1 <= 0) return cudaSuccess;
  dw_split(num_sms, tot0, tot1, &p.parts[0], &p.parts[1]);
  if (p.parts[0] + p.parts[1] < 1) return cudaSuccess;
  if (exact_grad) dw::dw_kernel<true><<<(p.parts[0] + p.parts[1]) * dw::kGroups, dw::kThreads, dw::kSmemBytes, st>>>(p);
  else dw::dw_kernel<false><<<(p.parts[0] + p.parts[1]) * dw::kGroups, dw::kThreads, dw::kSmemBytes, st>>>(p);
  ++*launches;
  return cudaGetLastError();
}

static int fin_numel_host(int t) {
  switch (t) {
    case 0: return 256 * 171;
    case 6: return 256 * 427;
    case 2: case 4: case 8: case 10: case 12: return 65536;
    case 1: case 3: case 5: case 7: case 9: case 11: case 13: case 14: return 256;
    case 15: return 1;
    case 16: return 128 * 280;
    case 18: case 20: return 128 * 128;
    case 17: case 19: case 21: return 128;
    case 24: return 3 * 128;
    case 25: return 3;
    default: return 0;
  }
}

// Chain rule through the folds for one or both networks + d latent, two launches in all.
cudaError_t launch_finalize_all(const float* const params_c[26], float* const grads_c[26], const float* acc_c,
                                const float* const params_f[26], float* const grads_f[26], const float* acc_f, const float* cond,
                                float* latent_out, cudaStream_t st, long long* launches) {
  FinAll f;
  f.nets = params_f ? 2 : 1;
  f.latent_out = latent_out;
  for (int i = 0; i < 26; ++i) {
    f.net[0].p[i] = params_c[i]; f.net[0].g[i] = grads_c[i];
    f.net[1].p[i] = params_f ? params_f[i] : nullptr; f.net[1].g[i] = params_f ? grads_f[i] : nullptr;
  }
  f.net[0].acc = acc_c; f.net[1].acc = acc_f;
  f.net[0].cond = f.net[1].cond = cond;
  int blocks = 1;  // + the latent block
  for (int t = 0; t < 26; ++t) blocks += (fin_numel_host(t) + 255) / 256;
  finalize_kernel<<<dim3(blocks, f.nets), 256, 0, st>>>(f);
  ++*launches;
  fin_dir0_kernel<<<dim3((128 * 256 + 256) * 32 / 256, f.nets), 256, 0, st>>>(f);
  ++*launches;
  return cudaGetLastError();
}

}  // namespace nfb
