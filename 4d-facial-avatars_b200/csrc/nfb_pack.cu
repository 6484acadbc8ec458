// nfb_pack.cu — load-time, per-optimizer-step and per-frame preparation kernels (not on the per-ray hot path):
//   * fold_feat_kernel : fc_feat pre-multiplied into fc_alpha and layers_dir.0[:, :256] (FP64 accumulate), both networks
//   * repack_kernel    : ONE launch per weight update, both networks: FP32 weights -> FP16 hi/lo as the swizzled shared-memory images the
//                        render kernels bulk-copy (forward streams) and the transposed streams of the backward chain (FP16 and hi/lo), static
//                        biases, conditioning columns, transposed direction columns
//   * frame_fold_kernel: per-frame expression/latent fold into the layer-0 / layer-3 biases
// Reference semantics: nerf/models.py:236-261 (forward), :218-233 (parameter shapes).
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "nfb_internal.h"
#include "nfb_layout.h"

namespace nfb {

// Folded step-6 matrix, computed where it is needed (FP64 accumulate, like a separate fold pass would):
//   W6[n][k], n < 128: (Wd0[:, :256] @ Wf)[n][k];  n == 128: (wa @ Wf)[k];  n > 128: 0
//   b6[n],    n < 128: bd0[n] + Wd0[n, :256] . bf;  n == 128: ba + wa . bf
struct NetParams { const float* p[26]; const float* w6; const float* b6; };  // state_dict order (nfb.h: nfb_load_weights) + the fold
// One quarter (j in [64 jq, 64 jq + 64)) of the dot product behind W6[n][k], four independent FP64 chains.
__device__ __forceinline__ double w6_quarter(const NetParams& a, int n, int k, int jq) {
  const float* left = (n < 128) ? (a.p[16] + (size_t)n * 280) : a.p[14];
  const float* Wf = a.p[12];
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll 4
  for (int j = 64 * jq; j < 64 * jq + 64; j += 4) {
#pragma unroll
    for (int q = 0; q < 4; ++q) acc[q] += (double)left[j + q] * (double)Wf[(j + q) * 256 + k];
  }
  return (acc[0] + acc[1]) + (acc[2] + acc[3]);
}
__device__ __forceinline__ float b6_elem(const NetParams& a, int n) {
  if (n > 128) return 0.f;
  const float* left = (n < 128) ? (a.p[16] + (size_t)n * 280) : a.p[14];
  const float* bf = a.p[13];
  double b = (n < 128) ? (double)a.p[17][n] : (double)a.p[15][0];
  for (int j = 0; j < 256; ++j) b += (double)left[j] * (double)bf[j];
  return (float)b;
}
// Launch 1 of a re-pack: W6 [144][256] and b6 [144] of up to two networks (blockIdx.z).  Block = row n (blockIdx.x) x 64 columns
// (blockIdx.y) x the four quarters of the 256-long dot product (threadIdx.x >> 6): short FP64 chains, Wf[j][k] coalesced over k,
// left[j] a warp broadcast; the quarters are summed in a fixed order through shared memory.
struct FoldArgs { NetParams net[2]; float* w6[2]; float* b6[2]; };
__global__ void __launch_bounds__(256) fold_feat_kernel(const FoldArgs f) {
  __shared__ double part[4][64];
  const NetParams& a = f.net[blockIdx.z];
  const int n = blockIdx.x, kq = threadIdx.x & 63, jq = threadIdx.x >> 6, k = blockIdx.y * 64 + kq;
  part[jq][kq] = (n <= 128) ? w6_quarter(a, n, k, jq) : 0.0;
  __syncthreads();
  if (jq == 0) f.w6[blockIdx.z][n * 256 + k] = (float)((part[0][kq] + part[1][kq]) + (part[2][kq] + part[3][kq]));
  if (threadIdx.x == 0 && blockIdx.y == 0) f.b6[blockIdx.z][n] = b6_elem(a, n);
}

// step -> (source parameter index, leading dimension, valid output rows); step 6 is the folded matrix
__device__ __forceinline__ int step_src(int s) { return s <= 5 ? 2 * s : (s == 7 ? 18 : (s == 8 ? 20 : 24)); }
__device__ __forceinline__ int step_ld(int s) { return s == 0 ? 171 : (s == 3 ? 427 : (s <= 6 ? 256 : 128)); }
__device__ __forceinline__ int step_rows(int s) { return s <= 5 ? 256 : (s == 6 ? 129 : (s == 9 ? 3 : 128)); }

// Forward streams: one thread per 16-byte chunk (8 consecutive K) of one weight row of unit `u` of step `s`.
__device__ __forceinline__ void pack_fwd_chunk(const NetParams& a, int s, int u, int idx, uint8_t* __restrict__ dst_x1,
                                               uint8_t* __restrict__ dst_x3) {
  const StepInfo si = step_info(s);
  if (u >= num_units(s)) return;
  const UnitInfo ui = unit_info(s, u);
  if (idx >= ui.rows * 8) return;
  const float* __restrict__ src = a.p[step_src(s)];
  const int ld = step_ld(s), n_valid = step_rows(s);
  const int c16 = idx & 7;
  const int n_local = idx >> 3;
  const int n = (ui.h ? si.nh0 : 0) + n_local;  // row of the step's logical weight matrix
  __align__(16) __half hi[8];
  __align__(16) __half lo[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int k = ui.ka * 64 + c16 * 8 + e;  // logical K index of this step
    float w = 0.f;
    if (n < n_valid) {
      if (s == 6) w = a.w6[n * 256 + k];
      else if (si.pe_first) {
        if (k < kDimXyz) w = src[(size_t)n * ld + k];
        else if (k >= 64) w = src[(size_t)n * ld + (kDimXyz + kDimCond) + (k - 64)];
      } else {
        w = src[(size_t)n * ld + k];
      }
    }
    hi[e] = __float2half_rn(w);
    lo[e] = __float2half_rn(w - __half2float(hi[e]));
  }
  const size_t unit_x1 = (size_t)step_offset_x1(s) + unit_offset_in_step(s, u);
  const int inner = n_local * 128 + ((c16 ^ (n_local & 7)) << 4);
  *reinterpret_cast<uint4*>(dst_x1 + unit_x1 + inner) = *reinterpret_cast<const uint4*>(hi);
  const size_t unit_x3 = 2 * unit_x1;
  *reinterpret_cast<uint4*>(dst_x3 + unit_x3 + inner) = *reinterpret_cast<const uint4*>(hi);
  *reinterpret_cast<uint4*>(dst_x3 + unit_x3 + (size_t)ui.rows * 128 + inner) = *reinterpret_cast<const uint4*>(lo);
}

// Static bias block, the 108 conditioning columns of layers_xyz.0/.3 and the transposed direction columns of layers_dir.0.
__device__ __forceinline__ void gather_elem(const NetParams& g, int t, float* __restrict__ bias_static, float* __restrict__ w0c,
                                            float* __restrict__ w3c, float* __restrict__ wd0b_t) {
  if (t < kBiasFloats) {
    float v = 0.f;
    if (t < 1536) v = g.p[2 * (t / 256) + 1][t % 256];       // layers_xyz.{0..5}.bias
    else if (t < 1680) v = g.b6[t - 1536];                    // folded layers_dir.0 / fc_alpha
    else if (t < 1808) v = g.p[19][t - 1680];                 // layers_dir.1.bias
    else if (t < 1936) v = g.p[21][t - 1808];                 // layers_dir.2.bias
    else if (t < 1939) v = g.p[25][t - 1936];                 // fc_rgb.bias
    bias_static[t] = v;
  }
  if (t < 256 * kDimCond) {
    const int n = t / kDimCond, j = t % kDimCond;
    w0c[t] = g.p[0][(size_t)n * 171 + kDimXyz + j];
    w3c[t] = g.p[6][(size_t)n * 427 + kDimXyz + j];
  }
  if (t < kDimDir * 128) {
    const int j = t / 128, n = t % 128;
    wd0b_t[t] = g.p[16][(size_t)n * 280 + 256 + j];  // layers_dir.0.weight[:, 256 + j]
  }
}

// Backward (transposed) streams: one thread per 16-byte chunk (8 consecutive k) of row n of unit (s, u); element (n, k) = W^T.
// dst: FP16 of W^T; dst_x3: hi then lo per unit (the split of the FP32 value, after the FP64 fold for M1 / m2).
__device__ __forceinline__ void pack_bwd_chunk(const NetParams& a, int s, int u, int idx, uint8_t* __restrict__ dst,
                                               uint8_t* __restrict__ dst_x3) {
  const StepInfo si = bwd_step_info(s);
  if (u >= si.k_atoms) return;
  const int rows = si.nh0 + si.nh1;
  if (idx >= rows * 8) return;
  const int c16 = idx & 7, n = idx >> 3;
  const bool op_atom = si.pe_first && u == 0;
  const int hid = u - si.pe_first;  // TMEM atom index
  __align__(16) __half h[8];
  __align__(16) __half lo[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int kl = c16 * 8 + e;        // k inside the atom
    const int kk = hid * 64 + kl;      // output-feature index of the forward layer (TMEM atoms)
    float w = 0.f;
    switch (s) {
      case 0: if (kl < 3) w = a.p[24][kl * 128 + n]; break;                       // fc_rgb.weight[kl][n]
      case 1: w = a.p[20][kk * 128 + n]; break;                                    // layers_dir.2.weight[kk][n]
      case 2: w = a.p[18][kk * 128 + n]; break;                                    // layers_dir.1
      case 3: if (op_atom) { if (kl == 3) w = a.w6[128 * 256 + n]; }               // m2 = fc_alpha . fc_feat
              else w = a.w6[kk * 256 + n]; break;                                  // M1 = layers_dir.0[:, :256] . fc_feat
      case 4: w = a.p[10][kk * 256 + n]; break;                                    // layers_xyz.5
      case 5: w = a.p[8][kk * 256 + n]; break;                                     // layers_xyz.4
      case 6: w = a.p[6][(size_t)kk * 427 + (kDimXyz + kDimCond) + n]; break;      // layers_xyz.3[:, 171:]
      case 7: w = a.p[4][kk * 256 + n]; break;                                     // layers_xyz.2
      default: w = a.p[2][kk * 256 + n]; break;                                    // layers_xyz.1
    }
    h[e] = __float2half_rn(w);
    lo[e] = __float2half_rn(w - __half2float(h[e]));
  }
  const int off = bwd_step_offset(s) + u * rows * 128;
  const int inner = n * 128 + ((c16 ^ (n & 7)) << 4);
  *reinterpret_cast<uint4*>(dst + off + inner) = *reinterpret_cast<const uint4*>(h);
  *reinterpret_cast<uint4*>(dst_x3 + 2 * off + inner) = *reinterpret_cast<const uint4*>(h);
  *reinterpret_cast<uint4*>(dst_x3 + 2 * off + rows * 128 + inner) = *reinterpret_cast<const uint4*>(lo);
}

// Launch 2 re-packs up to two networks: FP32 parameters (+ the fold) -> forward streams (x1, hi/lo x3), transposed backward
// stream, bias block, conditioning columns, direction columns.  Block ranges per network: [0, kFwdBlocks) forward chunks (8 blocks
// per (step, unit)), then backward chunks, then the gather.  Used by nfb_load_weights and by the fused optimizer step.
constexpr int kMaxFwdUnits = 5, kMaxBwdUnits = 4;
constexpr int kFwdBlocks = 8 * kMaxFwdUnits * kNumSteps;   // 400
constexpr int kBwdBlocks = 8 * kMaxBwdUnits * kBwdSteps;   // 288
constexpr int kGatherBlocks = (256 * kDimCond + 255) / 256;  // 108
constexpr int kRepackBlocks = kFwdBlocks + kBwdBlocks + kGatherBlocks;
struct RepackArgs {
  NetParams net[2];
  uint8_t *x1[2], *x3[2], *bwd[2], *bwd_x3[2];
  float *bias_static[2], *w0c[2], *w3c[2], *wd0b_t[2];
};
__global__ void __launch_bounds__(256) repack_kernel(const RepackArgs a) {
  const int net = blockIdx.y;
  int b = blockIdx.x;
  const NetParams& np = a.net[net];
  if (b < kFwdBlocks) {
    const int s = b / (8 * kMaxFwdUnits), r = b % (8 * kMaxFwdUnits);
    pack_fwd_chunk(np, s, r / 8, (r % 8) * 256 + threadIdx.x, a.x1[net], a.x3[net]);
    return;
  }
  b -= kFwdBlocks;
  if (b < kBwdBlocks) {
    const int s = b / (8 * kMaxBwdUnits), r = b % (8 * kMaxBwdUnits);
    pack_bwd_chunk(np, s, r / 8, (r % 8) * 256 + threadIdx.x, a.bwd[net], a.bwd_x3[net]);
    return;
  }
  b -= kBwdBlocks;
  gather_elem(np, b * 256 + threadIdx.x, a.bias_static[net], a.w0c[net], a.w3c[net], a.wd0b_t[net]);
}

// Per-frame conditioning in ONE launch.  Per network kFoldSlabs blocks: bias_frame = bias_static, then rows of step 0 and step 3
// += W[:, 63:171] . [expr/3 ; latent] (coalesced row loads, the accumulation order of a scalar loop).  One more block:
// cond[108] = [expr/3 ; latent] (the backward's chain rule through this fold needs it).
struct FrameFoldArgs {
  const float *bias_static[2], *w0c[2], *w3c[2];
  float* bias_frame[2];
  float* cond;
  int n_nets;
};
constexpr int kFoldSlabs = 8;  // blocks per network: 64 of the 512 folded bias rows each (one warp per row, lanes over the 108 columns)
__global__ void __launch_bounds__(256) frame_fold_kernel(const float* __restrict__ expr, const float* __restrict__ latent, const FrameFoldArgs a) {
  __shared__ float c[kDimCond];
  const int t = threadIdx.x;
  if (t < kDimExpr) c[t] = __fdiv_rn(expr[t], 3.0f);  // (expr * 1 / 3), models.py:241
  else if (t < kDimCond) c[t] = latent[t - kDimExpr];
  __syncthreads();
  const int net = blockIdx.x / kFoldSlabs, slab = blockIdx.x % kFoldSlabs;
  if (net >= a.n_nets) {
    if (slab == 0 && t < kDimCond) a.cond[t] = c[t];
    return;
  }
  const float* __restrict__ bias_static = a.bias_static[net];
  float* __restrict__ bias_frame = a.bias_frame[net];
  if (slab == 0)  // the entries no fold touches: steps 1, 2 and 4..9
    for (int i = t; i < kBiasFloats; i += blockDim.x)
      if (!(i < 256 || (i >= 768 && i < 1024))) bias_frame[i] = bias_static[i];
  const int warp = t >> 5, lane = t & 31;
  for (int r = warp; r < 64; r += 8) {
    const int row = slab * 64 + r;                 // 0..255: layers_xyz.0, 256..511: layers_xyz.3
    const int n = row & 255;
    const float* __restrict__ w = (row < 256 ? a.w0c[net] : a.w3c[net]) + n * kDimCond;
    // the same left-to-right fma chain a single thread would run (j ascending), split over lanes would change the rounding of
    // the per-frame bias by ~1 ulp; keep the sequential order: lane 0 accumulates, the other lanes only prefetch into registers
    float wv[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) wv[q] = (lane + 32 * q < kDimCond) ? w[lane + 32 * q] : 0.f;
    float acc = 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q)
      for (int l = 0; l < 32; ++l) {
        const float x = __shfl_sync(0xffffffffu, wv[q], l);
        if (l + 32 * q < kDimCond) acc = fmaf(x, c[l + 32 * q], acc);
      }
    const int bi = (row < 256) ? n : 768 + n;
    if (lane == 0) bias_frame[bi] = bias_static[bi] + acc;
  }
}

cudaError_t launch_repack(NetBuffers* const nb[2], const float* const* const params[2], int n_nets, cudaStream_t st,
                          long long* launches) {
  RepackArgs a;
  FoldArgs f;
  for (int n = 0; n < n_nets; ++n) {
    for (int i = 0; i < 26; ++i) { a.net[n].p[i] = params[n][i]; f.net[n].p[i] = params[n][i]; }
    f.net[n].w6 = f.net[n].b6 = nullptr;
    f.w6[n] = nb[n]->w6; f.b6[n] = nb[n]->b6;
    a.net[n].w6 = nb[n]->w6; a.net[n].b6 = nb[n]->b6;
    a.x1[n] = nb[n]->stream_x1; a.x3[n] = nb[n]->stream_x3; a.bwd[n] = nb[n]->stream_bwd; a.bwd_x3[n] = nb[n]->stream_bwd_x3;
    a.bias_static[n] = nb[n]->bias_static; a.w0c[n] = nb[n]->w0c; a.w3c[n] = nb[n]->w3c; a.wd0b_t[n] = nb[n]->wd0b_t;
  }
  fold_feat_kernel<<<dim3(144, 4, n_nets), 256, 0, st>>>(f);
  ++*launches;
  repack_kernel<<<dim3(kRepackBlocks, n_nets), 256, 0, st>>>(a);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_frame_fold(NetBuffers* const nb[2], int n_nets, const float* expr, const float* latent, float* cond,
                              cudaStream_t st, long long* launches) {
  FrameFoldArgs a;
  for (int n = 0; n < n_nets; ++n) {
    a.bias_static[n] = nb[n]->bias_static; a.w0c[n] = nb[n]->w0c; a.w3c[n] = nb[n]->w3c; a.bias_frame[n] = nb[n]->bias_frame;
  }
  a.cond = cond;
  a.n_nets = n_nets;
  frame_fold_kernel<<<(n_nets + 1) * kFoldSlabs, 256, 0, st>>>(expr, latent, a);
  ++*launches;
  return cudaGetLastError();
}

}  // namespace nfb
