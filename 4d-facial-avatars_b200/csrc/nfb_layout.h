// nfb_layout.h — the MLP as the kernel executes it: 10 tensor-core "steps", each a GEMM
//   D[128 rows, N] = A[128 rows, K] * W[N, K]^T   (FP16 operands, FP32 accumulate in TMEM)
// and the byte layout of the packed weight stream the kernel bulk-copies into shared memory.
// Shared by host (packing, tests) and device code.
//
// Reference model: ConditionalBlendshapePaperNeRFModel.forward (nerf/models.py:236-261).  Exact
// algebra applied at load / per frame (SURVEY.md §8 a''):
//   * the 108 expression/latent columns of layers_xyz.0 and layers_xyz.3 multiply a per-frame constant
//     vector -> folded into those layers' biases (nfb_set_frame);
//   * fc_feat has no activation -> pre-multiplied into fc_alpha and layers_dir.0[:, :256] (FP64 fold);
//   * the 24 direction-encoding columns of layers_dir.0 depend on the ray only -> a per-ray bias.
//
//   step  reference layer            N (half 0 + half 1)  K (atoms of 64)            A operand
//   0     layers_xyz.0               128 + 128            64  = PE(63)+pad           SMEM (PE buffer)
//   1,2   layers_xyz.1,2             128 + 128            256                        TMEM
//   3     layers_xyz.3               128 + 128            320 = PE(63)+pad | h(256)  SMEM atom + TMEM
//   4,5   layers_xyz.4,5             128 + 128            256                        TMEM
//   6     layers_dir.0∘fc_feat | σ   128 + 16 (σ)         256                        TMEM
//   7,8   layers_dir.1,2             128                  128                        TMEM
//   9     fc_rgb                     16 (3 used)          128                        TMEM
//
// A weight "unit" = all N rows of the step x one 64-wide K atom (<= 32 KB), consumed by 4 tcgen05.mma (M=128, N, K=16).
// The epilogue converts the accumulator in two column halves ("half 0" = output columns [0,128) = K atoms 0,1 of the
// next step, "half 1" = [128,256) = atoms 2,3) and signals each; the units of the next step are grouped by what they
// need:   [PE atom] [hidden atoms 0,1] = group 1 (needs half 0 only)   |   [hidden atoms 2,3] = group 2 (needs half 1 too)
// so the next step starts on atoms 0,1 while the second half of the previous step is still being converted.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define NFB_HD __host__ __device__
#else
#define NFB_HD
#endif

namespace nfb {

constexpr int kTileM = 128;      // rows (samples) per tensor-core tile == TMEM lanes
constexpr int kAtomK = 64;       // fp16 elements per 128-byte swizzle row
constexpr int kNumSteps = 10;
constexpr int kMaxUnitBytes = 256 * 128;  // one weight unit: <=256 output rows x 64 K x 2 B
constexpr int kDimXyz = 63, kDimDir = 24, kDimExpr = 76, kDimLatent = 32, kDimCond = 108;

struct StepInfo {
  int16_t nh0, nh1;   // output columns (= MMA N) of half 0 / half 1; nh1 == 0: single half
  int16_t k_atoms;    // K / 64 including the PE atom
  int16_t pe_first;   // 1: the first K atom is the positional encoding (A from shared memory)
  int16_t bias_off;   // float offset of this step's bias vector in the per-network bias block
  int16_t n_bias;     // bias floats
};

NFB_HD constexpr StepInfo step_info(int s) {
  return s == 0   ? StepInfo{128, 128, 1, 1, 0, 256}
         : s == 1 ? StepInfo{128, 128, 4, 0, 256, 256}
         : s == 2 ? StepInfo{128, 128, 4, 0, 512, 256}
         : s == 3 ? StepInfo{128, 128, 5, 1, 768, 256}
         : s == 4 ? StepInfo{128, 128, 4, 0, 1024, 256}
         : s == 5 ? StepInfo{128, 128, 4, 0, 1280, 256}
         : s == 6 ? StepInfo{128, 16, 4, 0, 1536, 144}
         : s == 7 ? StepInfo{128, 0, 2, 0, 1680, 128}
         : s == 8 ? StepInfo{128, 0, 2, 0, 1808, 128}
                  : StepInfo{16, 0, 2, 0, 1936, 16};
}
constexpr int kBiasFloats = 1952;  // 6*256 + 144 + 128 + 128 + 16

// Bytes of the FP16 "hi" weights of one step (x1 stream); the x3 stream stores hi then lo per unit.
NFB_HD constexpr int step_bytes_x1(int s) {
  return (step_info(s).nh0 + step_info(s).nh1) * step_info(s).k_atoms * 128;
}
NFB_HD constexpr int step_offset_x1(int s) {
  int off = 0;
  for (int i = 0; i < s; ++i) off += step_bytes_x1(i);
  return off;
}
constexpr int kStreamBytesX1 = step_offset_x1(kNumSteps);  // 864256
constexpr int kStreamBytesX3 = 2 * kStreamBytesX1;

// The u-th weight unit of step s in consumption order.
struct UnitInfo {
  int16_t h;        // N-half (0/1): accumulator half and row block [h ? nh0 : 0, ...) of the layer's weight matrix
  int16_t ka;       // K atom of the step's logical K axis (0 = the PE atom when the step has one)
  int16_t from_pe;  // A operand comes from the shared-memory PE buffer
  int16_t group;    // 1: needs the previous step's half-0 epilogue only; 2: also its half-1 epilogue
  int16_t rows;     // output rows (MMA N) of the unit
  int16_t last;     // last unit of its half in this step (-> commit "accumulator half complete")
};
NFB_HD constexpr int num_units(int s) { return step_info(s).k_atoms; }
NFB_HD constexpr UnitInfo unit_info(int s, int u) {
  const StepInfo si = step_info(s);
  const int hid = u - si.pe_first;  // hidden atom index (< 0: the PE atom)
  const int group = (hid >= 2) ? 2 : 1;
  return UnitInfo{0, (int16_t)u, (int16_t)(si.pe_first && u == 0), (int16_t)group, (int16_t)(si.nh0 + si.nh1),
                  (int16_t)(u == si.k_atoms - 1)};
}
// Byte offset of unit u inside its step, x1 stream.
NFB_HD constexpr int unit_offset_in_step(int s, int u) {
  int off = 0;
  for (int i = 0; i < u; ++i) off += unit_info(s, i).rows * 128;
  return off;
}
// Byte offset of element (row n, k in [0,64)) inside one swizzled unit: 128-byte rows, 16-byte chunks
// XORed with (row & 7) — the SWIZZLE_128B pattern the UMMA shared-memory descriptor expects.
NFB_HD constexpr int sw128_offset(int n, int k) { return n * 128 + ((((k >> 3) ^ (n & 7)) & 7) << 4) + ((k & 7) << 1); }


// ------------------------------------------------------------------------------------------------
// Training: per-tile activation record (written by the forward kernel in SAVE mode and by the backward chain kernel,
// read by the weight-gradient kernel).  Every entry is a TRANSPOSED image of a [128 sample rows x C features] FP16
// matrix: element (feature k, sample r) lives in r-atom (r >> 6) — a [C rows x 64 r] block in the same 128-byte-swizzled
// K-major layout as a weight unit — so the weight-gradient GEMM  dW[n,k] = sum_r dY[r,n] X[r,k]  reads both operands
// with plain bulk copies and the K-major descriptors of the forward pass (reduction dimension = sample rows).
constexpr int kRecPE = 0;                         // positional encoding, 64 features (lane 63 = 0)
constexpr int kRecH0 = 16384;                     // h0..h5 (outputs of tensor-core steps 0..5), 256 features each
constexpr int kRecG0 = kRecH0 + 6 * 65536;        // g0..g2 (steps 6..8), 128 features each
constexpr int kRecPEd = kRecG0 + 3 * 32768;       // per-ray direction encoding replicated per sample, 32 rows (24 used)
constexpr int kRecMask = kRecPEd + 8192;          // ReLU masks: [9 layers][128 rows][8 x u32]
constexpr int kRecDY0 = kRecMask + 9 * 128 * 32;  // dY0..dY5 (gradient w.r.t. the pre-activation of steps 0..5), 256 features
constexpr int kRecDY6 = kRecDY0 + 6 * 65536;      // dY6..dY8, 128 features
constexpr int kRecDRaw = kRecDY6 + 3 * 32768;     // scaled (d rgb_raw[3], d sigma_raw) image, 16 rows (4 used)
constexpr int kRecBytes = kRecDRaw + 4096;
static_assert(kRecBytes == (1 << 20), "tile record is 1 MiB");
// Exact-gradient training (NFB_PREC_EXACT_GRAD): a tile record is 2 MiB.  The first MiB is the record above, byte for byte; the
// second holds the lo parts  lo = fp16(x - float(hi))  of every image at the same offsets (PE, h0..h5, g0..g2, PEd, dY0..dY8,
// dRaw), so x = hi + lo to ~2^-21 relative.  The mask region of the lo MiB is unused.
constexpr int kRecLo = 1 << 20;
NFB_HD constexpr long long rec_stride(bool exact_grad) { return exact_grad ? 2LL * kRecBytes : (long long)kRecBytes; }
NFB_HD constexpr int rec_x_off(int layer) { return layer < 6 ? kRecH0 + layer * 65536 : kRecG0 + (layer - 6) * 32768; }
NFB_HD constexpr int rec_dy_off(int layer) { return layer < 6 ? kRecDY0 + layer * 65536 : kRecDY6 + (layer - 6) * 32768; }
NFB_HD constexpr int rec_width(int layer) { return layer < 6 ? 256 : 128; }
// Byte offset of element (feature k, sample row r) inside an image with `rows` features.
NFB_HD constexpr int img_offset(int rows, int k, int r) { return (r >> 6) * rows * 128 + sw128_offset(k, r & 63); }

// Backward chain (dX): 9 tensor-core steps per 128-row tile, same machinery as the forward pass with transposed weights.
//   step  computes                         N (half0+half1)  K atoms                A operand
//   0     d g2 = d rgb . Wrgb              128              1 (smem, k<3 used)     SMEM (d raw operand)
//   1     d g1 = dY8 . Wd2                 128              2                      TMEM
//   2     d g0 = dY7 . Wd1                 128              2                      TMEM
//   3     d h5 = dY6 . M1 + d sigma . m2   128 + 128        1 (smem, k=3) + 2      SMEM atom + TMEM
//   4..8  d h4..h0 = dY . W5, W4, W3[:,171:], W2, W1   128 + 128   4               TMEM
// The epilogue of step s multiplies by the ReLU mask of forward layer (8 - s) and yields dY(8 - s).
constexpr int kBwdSteps = 9;
NFB_HD constexpr StepInfo bwd_step_info(int s) {
  return s == 0   ? StepInfo{128, 0, 1, 1, 0, 0}
         : s <= 2 ? StepInfo{128, 0, 2, 0, 0, 0}
         : s == 3 ? StepInfo{128, 128, 3, 1, 0, 0}
                  : StepInfo{128, 128, 4, 0, 0, 0};
}
NFB_HD constexpr int bwd_step_bytes(int s) { return (bwd_step_info(s).nh0 + bwd_step_info(s).nh1) * bwd_step_info(s).k_atoms * 128; }
NFB_HD constexpr int bwd_step_offset(int s) {
  int off = 0;
  for (int i = 0; i < s; ++i) off += bwd_step_bytes(i);
  return off;
}
constexpr int kBwdStreamBytes = bwd_step_offset(kBwdSteps);  // 835584
constexpr int kBwdStreamBytesX3 = 2 * kBwdStreamBytes;       // exact-gradient chain: per unit the hi image, then the lo image

// Weight-gradient accumulators of one network (FP32, float offsets), in the kernel's folded parametrisation.
constexpr int kAcc0 = 0;                       // [256][64]   d W0[:, PE lanes]
constexpr int kAcc1 = kAcc0 + 256 * 64;        // [256][256]
constexpr int kAcc2 = kAcc1 + 65536;
constexpr int kAcc3a = kAcc2 + 65536;          // [256][64]   d W3[:, PE lanes]
constexpr int kAcc3b = kAcc3a + 256 * 64;      // [256][256]  d W3[:, 171:427]
constexpr int kAcc4 = kAcc3b + 65536;
constexpr int kAcc5 = kAcc4 + 65536;
constexpr int kAcc6 = kAcc5 + 65536;           // [128][256]  d M1 (layers_dir.0[:, :256] . fc_feat)
constexpr int kAcc6d = kAcc6 + 128 * 256;      // [128][32]   d layers_dir.0[:, 256:280]
constexpr int kAccSig = kAcc6d + 128 * 32;     // [256][16]   column 3 = d m2 (fc_alpha . fc_feat)
constexpr int kAcc7 = kAccSig + 256 * 16;      // [128][128]
constexpr int kAcc8 = kAcc7 + 128 * 128;
constexpr int kAcc9 = kAcc8 + 128 * 128;       // [128][16]   transposed: [k][n], n < 3 = d fc_rgb.weight[n][k]
constexpr int kAccB = kAcc9 + 128 * 16;        // biases: b0..b5 [256] each, b6..b8 [128] each, then [4] = (d b_rgb[3], d b_sigma)
constexpr int kAccBRaw = kAccB + 6 * 256 + 3 * 128;
constexpr int kAccFloats = kAccBRaw + 4;
NFB_HD constexpr int acc_bias_off(int layer) { return kAccB + (layer < 6 ? layer * 256 : 1536 + (layer - 6) * 128); }

// Algorithmic cost used for the roofline (SURVEY.md §8d): 550,016 MAC per MLP evaluation.
constexpr long long kAlgoFlopPerEval = 1100032LL;
// MACs the kernel actually issues per evaluation after the folds above.
constexpr long long kExecMacPerEval = 64LL * 256 + 4LL * 256 * 256 + 320LL * 256 + 256LL * 144 + 2LL * 128 * 128 + 128LL * 16;

}  // namespace nfb
