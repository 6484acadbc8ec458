// nfb_internal.h — structures shared between the C-ABI layer (nfb_api.cu), the preparation kernels
// (nfb_pack.cu) and the render kernel (nfb_render.cu).  Not part of the public interface.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "nfb_sampler.h"

namespace nfb {

// Device buffers of one loaded network.
struct NetBuffers {
  uint8_t* stream_x1 = nullptr;  // kStreamBytesX1: FP16 weights, swizzled units in execution order
  uint8_t* stream_x3 = nullptr;  // kStreamBytesX3: hi unit, lo unit, ...
  float* w6 = nullptr;           // [144,256] folded layers_dir.0 / fc_alpha
  float* b6 = nullptr;           // [144]
  float* bias_static = nullptr;  // [kBiasFloats]
  float* bias_frame = nullptr;   // [kBiasFloats] bias_static + per-frame fold (what the kernel reads)
  float* w0c = nullptr;          // [256,108] conditioning columns of layers_xyz.0
  float* w3c = nullptr;          // [256,108] conditioning columns of layers_xyz.3
  float* wd0b_t = nullptr;       // [24,128] direction columns of layers_dir.0, transposed
  uint8_t* stream_bwd = nullptr; // kBwdStreamBytes: transposed FP16 weights for the backward chain (nfb_train.cu)
  uint8_t* stream_bwd_x3 = nullptr;  // kBwdStreamBytesX3: the same as hi unit, lo unit, ... (exact-gradient chain)
  bool loaded = false;
};

// Everything the render kernel needs, passed by value (__grid_constant__).
struct RenderParams {
  // rays
  const float* o;
  const float* d;
  int n_rays;
  float pose[12];
  float fx, fy, wcx, hcy;  // intrinsics as FP32; wcx = width*cx, hcy = height*cy (rounded like torch does)
  int width, row_begin;
  float near_, far_;
  const float* dir_z;
  const float* bg;
  // sampling
  int nc, nf, s_fine;     // s_fine = nc + nf
  int rays_per_unit;      // R
  int tiles_c, tiles_f;   // 128-row tiles per coarse / fine pass of one unit
  int n_units;
  int perturb;
  float noise_std;
  int white_bkgd;
  const float* t_coarse;  // [nc]
  const float* u_fine;    // [nf]
  const float *t_rand, *noise_c, *u_rand, *noise_f;
  // networks
  const uint8_t* wstream[2];
  const float* bias[2];
  const float* wd0b_t[2];
  // outputs
  float *rgb_c, *disp_c, *acc_c, *rgb_f, *disp_f, *acc_f, *w_last;
  // training forward (all null in evaluation): per-tile activation records (nfb_layout.h kRec*), per-ray |d|, and per
  // sample (colour or bg, ReLU input of sigma) of both passes
  uint8_t* save_rec;
  float* save_dnorm;
  float *save_raw_c, *save_raw_f;
  // debug
  float *dbg_z_c, *dbg_raw_c, *dbg_z_f, *dbg_raw_f, *dbg_act;
  int dbg_act_step;
  unsigned long long* prof;  // optional [64] phase-cycle counters (see PhaseTimer in nfb_render.cu)
};

// ---- training (nfb_train.cu)
struct CompBwdParams {
  int n_rays, nc, nf, s_fine, rays_per_unit, tiles_c, tiles_f, has_bg, white_bkgd;
  const float *z_c, *raw_c, *z_f, *raw_f, *dnorm;                       // saved by the training forward
  const float *g_rgb[2], *g_disp[2], *g_acc[2], *g_wlast;               // dL/d outputs (coarse, fine); any may be null
  float* draw;                                                          // [tiles][128][4] dL/d(rgb_raw, sigma_raw), zero-initialised
  float* acc[2];                                                        // per-network accumulators (kAccBRaw sums land here)
  unsigned int* absmax;                                                 // max |d raw| as float bits
};
struct ChainParams {
  int n_units, tiles_c, tiles_f;
  uint8_t* rec;
  const float* draw;
  const float* scal;            // [0] = loss scale, [1] = 1 / scale
  const uint8_t* wstream[2];    // backward weight streams (coarse, fine): stream_bwd, or stream_bwd_x3 for the exact-gradient chain
};
struct DwParams {  // ONE launch covers both networks: the first parts[0] * groups CTAs work on network 0, the rest on network 1
  const uint8_t* rec;
  int n_units, tpu;
  int t_base[2], t_cnt[2];  // tiles of network i: unit * tpu + t_base[i] + [0, t_cnt[i])
  int parts[2];             // CTAs per job group of network i (set by launch_dw, proportional to the tile counts)
  float* acc[2];
  const float* scal;
};
// host copies of the compile-time schedules (nfb_debug_schedule); index < 0: number of entries; else words written or -1
int debug_prog_v4(int index, uint32_t* out);
int debug_prog_v6(int index, uint32_t* out);
int debug_jobs_v7(int n_iter, int tc, int tf, int index, uint32_t* out);
int debug_prog_chain(int index, uint32_t* out);
int debug_jobs_dw(int index, uint32_t* out);
int debug_prog_chain_exact(int index, uint32_t* out);
int debug_stages_dw_exact(int index, uint32_t* out);
int debug_dw_split(uint32_t* io);  // io: {num_sms, tiles net 0, tiles net 1} -> {parts0, parts1, groups}
cudaError_t train_kernels_setup();
cudaError_t launch_composite_bwd(const CompBwdParams& q, float* scal, cudaStream_t st, long long* launches);
// exact_grad: the variants that read / write 2 MiB hi+lo records (after an NFB_PREC_EXACT_GRAD training forward)
cudaError_t launch_chain(const ChainParams& p, bool exact_grad, int num_sms, cudaStream_t st, long long* launches);
cudaError_t launch_dw(const DwParams& p, bool exact_grad, int num_sms, cudaStream_t st, long long* launches);
cudaError_t launch_finalize_all(const float* const params_c[26], float* const grads_c[26], const float* acc_c,
                                const float* const params_f[26], float* const grads_f[26], const float* acc_f, const float* cond,
                                float* latent_out, cudaStream_t st, long long* launches);

// Two launches (fold, pack): FP32 parameters of n_nets (1 or 2) networks -> forward / backward weight streams, bias block, conditioning and
// direction columns (nfb_pack.cu: repack_kernel).
cudaError_t launch_repack(NetBuffers* const nb[2], const float* const* const params[2], int n_nets, cudaStream_t st, long long* launches);
// One launch: per-frame bias fold of the loaded networks + cond[108] = [expr / 3 ; latent].
cudaError_t launch_frame_fold(NetBuffers* const nb[2], int n_nets, const float* expr, const float* latent, float* cond,
                              cudaStream_t st, long long* launches);
// Training-step tail (nfb_optim.cu): d mse / d rgb (+ loss sums), Adam over a flat bucket with zero_grad fused.
cudaError_t launch_loss_grad(const float* rgb_c, const float* rgb_f, const float* target, int n_rays, long long n_total, float* g_c,
                             float* g_f, float* loss, cudaStream_t st, long long* launches);
cudaError_t launch_adam_dev(float* p, float* g, float* m, float* v, long long n, void* dev_state, cudaStream_t st, long long* launches);
cudaError_t launch_adam(float* p, float* g, float* m, float* v, long long n, float lr, float b1, float b2, float eps, int step,
                        float grad_scale, long long reg_off, float reg_w, cudaStream_t st, long long* launches);
// precision: 0 = fast (x1), 1 = exact (x3), 2 = exact with lo records (training forward of NFB_PREC_EXACT_GRAD; evaluation as 1).
// num_sms = CTAs to launch at most.
cudaError_t launch_render(const RenderParams& p, int precision, int num_sms, cudaStream_t st, long long* launches);
cudaError_t render_kernel_setup();  // opt-in to the large dynamic shared memory size
// Two-tiles-in-flight kernel (nfb_render2.cu): fast-mode evaluation (the training forward and the layer probe run launch_render).
cudaError_t render2_kernel_setup();
cudaError_t launch_render2(const RenderParams& p, int num_sms, cudaStream_t st, long long* launches);
// Two tiles in flight + software-pipelined passes (nfb_render3.cu): fast-mode evaluation of the configurations its fixed
// shared-memory budget covers (render3_supports), bit-identical to nfb_render2.cu.
cudaError_t render3_kernel_setup();
bool render3_supports(const RenderParams& p);
cudaError_t launch_render3(const RenderParams& p, int num_sms, cudaStream_t st, long long* launches);

// ---- either side of the path (nfb_post.cu)
cudaError_t launch_frame_products(const float* rgb, const float* disp, const float* w_last, const double intr[4], int H, int W,
                                  uint8_t* rgb_u8, uint8_t* normals_u8, uint8_t* disp_u8, uint32_t* minmax_scratch, int like_torch_cpu,
                                  cudaStream_t st, long long* launches);
constexpr int kSmpMax = 2048;  // rays per sampler call (num_random_rays of the shipped YAML)
struct SampleArgs {
  smp::Map map;
  const double* draws;   // uniform [0,1) doubles, consumed like RandomState.rand: round r takes (size - n_found) values
  int size, max_rounds;
  long long* found;      // [size] selected flat indices in selection order (= np.random.choice's return value)
  int* state;            // [0] n_found, [1] rounds run, [2] draws consumed  (in/out: a call may resume a partial selection)
  smp::Run* runs;
  smp::Seg* segs;
  int* first_pos;        // [H * W] scratch, all INT_MAX between calls
  // gathers (any output may be null)
  float pose[12];
  float fx, fy, wcx, hcy;
  const float* image;       // [H, W, 3]
  const float* background;  // [H, W, 3]
  float *ray_o, *ray_d, *target, *bg_out;  // [size, 3] each
  int* pixel_rc;            // [size, 2] (row, col) of the selected pixels
};

cudaError_t launch_sample_rays(const SampleArgs& a, cudaStream_t st, long long* launches);
cudaError_t launch_fill_int(int* p, long long n, int v, cudaStream_t st, long long* launches);

}  // namespace nfb
