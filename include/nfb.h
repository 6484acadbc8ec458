/* nfb.h — C ABI of the B200-native NeRFace render path ("nfb" = NeRFace on Blackwell).
 *
 * This is the drop-in boundary for ONE hot path of gafniguy/4D-Facial-Avatars: the per-ray render
 * loop reached through nerface_code/nerf-pytorch/nerf/train_utils.py (run_one_iter_of_nerf :165-290,
 * predict_and_render_radiance :36-162, run_network :9-33), nerf_helpers.py (get_ray_bundle :68-123,
 * positional_encoding :195-239, sample_pdf_2 :344-387, cumprod_exclusive :44-65),
 * volume_rendering_utils.py (volume_render_radiance_field :7-75) and models.py
 * (ConditionalBlendshapePaperNeRFModel :189-261).  The reference has no FFI (it is pure PyTorch);
 * the Python package 4d-facial-avatars_b200/nerf binds these entry points with ctypes and keeps the
 * reference's call surface.  See INTEGRATION.md.
 *
 * Conventions: plain pointers and sizes, no torch types.  Every entry returns an int status
 * (0 = NFB_OK) and never throws; nfb_strerror() maps it to text.  All device pointers are FP32,
 * row-major, 16-byte aligned, on the device the handle was created for.  Calls are asynchronous on
 * the given cudaStream_t (passed as void*) unless stated otherwise; no entry synchronises the device
 * except nfb_render_frame_host.
 */
#ifndef NFB_H_
#define NFB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NFB_VERSION 121

typedef struct NfbHandle NfbHandle;

enum {
  NFB_OK = 0,
  NFB_ERR_INVALID = 1,     /* bad argument (null pointer, negative size, ...) */
  NFB_ERR_UNSUPPORTED = 2, /* configuration outside what the kernel implements */
  NFB_ERR_CUDA = 3,        /* a CUDA runtime call failed; see nfb_last_cuda_error() */
  NFB_ERR_STATE = 4,       /* call order violated (weights or frame not set) */
  NFB_ERR_ARCH = 5         /* device is not sm_100 */
};

/* Which of the two networks (models.coarse / models.fine in the reference YAML). */
enum { NFB_NET_COARSE = 0, NFB_NET_FINE = 1 };

/* Arithmetic used by the tensor-core MLP.
 *   NFB_PREC_FAST       : FP16 operands (round-to-nearest), FP32 accumulate, one tcgen05 pass.
 *   NFB_PREC_EXACT      : every operand split x = hi + lo in FP16; hi*hi + hi*lo + lo*hi, FP32
 *                         accumulate (3 tcgen05 passes, ~2^-21 relative operand error).  In training
 *                         only the forward: nfb_render_backward carries FP16 operands (~2^-11).
 *   NFB_PREC_EXACT_GRAD : NFB_PREC_EXACT for rendering (same kernel, bit-identical outputs); after a
 *                         nfb_render_forward_train in this mode the backward's dX chain and weight-gradient
 *                         GEMMs use split operands as well (hi+lo records, see nfb_render_forward_train). */
enum { NFB_PREC_FAST = 0, NFB_PREC_EXACT = 1, NFB_PREC_EXACT_GRAD = 2 };

/* Encoder / conditioning dimensions; mirrors the constructor arguments of
 * ConditionalBlendshapePaperNeRFModel (models.py:193-206).  Only the shipped paper configuration
 * (10, 4, include_input_xyz=1, include_input_dir=0, 76, 32) is implemented. */
typedef struct {
  int32_t num_encoding_fn_xyz;
  int32_t num_encoding_fn_dir;
  int32_t include_input_xyz;
  int32_t include_input_dir;
  int32_t dim_expression;
  int32_t dim_latent;
} NfbModelDims;

/* Rays of one call.  Either explicit rays (o and d non-null; what run_one_iter_of_nerf receives,
 * train_utils.py:171-172) or in-kernel generation from a camera (o == d == NULL; replaces
 * get_ray_bundle, nerf_helpers.py:68-123, for image rows [row_begin, row_begin + n_rays / width)). */
typedef struct {
  const float* o;          /* [n_rays,3] device, or NULL */
  const float* d;          /* [n_rays,3] device, unnormalised, or NULL */
  int32_t n_rays;
  float pose[12];          /* row-major 3x4 camera-to-world (used when o == NULL) */
  double intrinsics[4];    /* fx, fy, cx, cy with cx, cy relative in [0,1]; FP64 like the reference's numpy
                              array (load_flame.py:114-118), rounded to FP32 where torch would */
  int32_t height, width, row_begin;
  float near_, far_;       /* options.dataset.near / far (train_utils.py:210-211) */
  const float* dir_z;      /* optional [n_rays]: overrides d_z as the first input of the direction
                              encoder (ray_directions_ablation path, train_utils.py:81-82); NULL = d_z */
  const float* background; /* optional [n_rays,3] background_prior (train_utils.py:95-96) or NULL */
} NfbRays;

/* options.nerf.<mode>.* (train_utils.py:56-69,108-122). */
typedef struct {
  int32_t num_coarse, num_fine;
  int32_t perturb;          /* stratified coarse samples; also makes the fine resampling stochastic */
  float noise_std;          /* radiance_field_noise_std */
  int32_t white_background;
  int32_t lindisp;          /* must be 0 (all shipped YAMLs) */
  int32_t precision;        /* NFB_PREC_* */
  const float* t_coarse;    /* optional device [num_coarse] = torch.linspace(0,1,num_coarse); NULL: computed */
  const float* u_fine;      /* optional device [num_fine]  = torch.linspace(0,1,num_fine);  NULL: computed */
} NfbSampling;

/* Explicit noise, in the reference's draw order per ray chunk (SURVEY.md §8c).  Required members:
 * t_rand and u when perturb != 0; sigma_noise_* when noise_std > 0.  All device pointers. */
typedef struct {
  const float* t_rand;        /* [n_rays, num_coarse] uniform [0,1) */
  const float* sigma_noise_c; /* [n_rays, num_coarse] standard normal */
  const float* u;             /* [n_rays, num_fine] uniform [0,1) */
  const float* sigma_noise_f; /* [n_rays, num_coarse+num_fine] standard normal */
} NfbNoise;

/* The 7-tuple of predict_and_render_radiance (train_utils.py:162).  Fine members may be NULL when
 * num_fine == 0; then w_last receives the coarse pass's last weight. */
typedef struct {
  float* rgb_coarse;  /* [n_rays,3] */
  float* disp_coarse; /* [n_rays] */
  float* acc_coarse;  /* [n_rays] */
  float* rgb_fine;    /* [n_rays,3] */
  float* disp_fine;   /* [n_rays] */
  float* acc_fine;    /* [n_rays] */
  float* w_last;      /* [n_rays] weights[:, -1] of the last pass */
} NfbOutputs;

/* Optional per-sample dumps (tests, and the tensors a backward pass needs).  Any member may be NULL. */
typedef struct {
  float* z_coarse;   /* [n_rays, num_coarse] */
  float* raw_coarse; /* [n_rays, num_coarse, 4] MLP output (rgb raw, sigma raw), before the bg overwrite */
  float* z_fine;     /* [n_rays, num_coarse+num_fine] sorted */
  float* raw_fine;   /* [n_rays, num_coarse+num_fine, 4] */
  /* Layer probe: post-activation FP32 values the epilogue of tensor-core step `act_step` (0..8, see
   * nfb_layout.h; -1 = the 64-lane positional encoding) produced for the first 128 coarse rows
   * (rays 0.., samples in order).  [128, 256] floats; columns beyond the step's width are untouched. */
  float* act_dump;
  int32_t act_step;
  /* Phase timers: 64 uint64 cycle counters (zeroed by the caller), accumulated over all CTAs by one observer
   * thread per warp role.  Slots: 0 ray setup, 1 per-ray direction term, 2 sampling+encoding (prologue),
   * 10+s wait for tensor-core step s, 20+s epilogue of step s, 3 end-of-pass barrier, 4 compositing,
   * 5 cdf, 6 inverse-cdf sampling, 7 sort; 41 producer waiting for a free ring slot; 45 MMA issuer waiting for
   * the A operand, 46 waiting for weights, 44 issuing. */
  unsigned long long* prof;
} NfbDebug;

int nfb_version(void);
const char* nfb_strerror(int status);
/* Text of the last CUDA error seen by this thread's calls (empty string if none). */
const char* nfb_last_cuda_error(void);

/* Create / destroy a renderer bound to one CUDA device.  Allocates the packed-weight streams,
 * per-frame constant buffers and per-CTA scratch (a few MB). */
int nfb_create(const NfbModelDims* dims, int device, NfbHandle** out);
int nfb_destroy(NfbHandle* h);

/* Load one network.  `params` holds 26 DEVICE pointers in the reference's state_dict order
 * (models.py:218-233): layers_xyz.{0..5}.{weight,bias}, fc_feat.{weight,bias}, fc_alpha.{weight,bias},
 * layers_dir.{0..3}.{weight,bias}, fc_rgb.{weight,bias} — weights row-major (out,in).  Folds fc_feat
 * into fc_alpha / layers_dir.0 (exact algebra, FP64), splits to FP16 hi/lo and writes the
 * shared-memory-image weight streams the kernel's bulk copies read.  layers_dir.3 is ignored, as in
 * the reference's forward (models.py:257). */
int nfb_load_weights(NfbHandle* h, int which, const float* const params[26], void* stream);

/* Per-frame conditioning: expression[76] (divided by 3 inside, models.py:241) and latent[32], both
 * DEVICE pointers.  Folds W0[:,63:171]·c and W3[:,63:171]·c into the layer-0 / layer-3 biases of both
 * loaded networks. */
int nfb_set_frame(NfbHandle* h, const float* expression, const float* latent, void* stream);

/* The hot path: coarse sampling -> encode -> coarse MLP -> composite -> inverse-CDF resample -> sort
 * -> encode -> fine MLP -> composite, one persistent sm_100a kernel launch. */
int nfb_render_forward(NfbHandle* h, const NfbRays* rays, const NfbSampling* sampling,
                       const NfbNoise* noise /* nullable */, const NfbOutputs* out,
                       const NfbDebug* dbg /* nullable */, void* stream);

/* ---- Training (replaces torch.autograd over the unfused graph, train_transformed_rays.py:389) ----
 * nfb_render_forward_train is nfb_render_forward that additionally keeps, in buffers owned by the handle, what the
 * backward needs: per-sample depths, colours and ReLU inputs of both passes, and per 128-row tile the FP16 activations
 * of every layer (about 1 MiB per tile; 2048 rays at 64+64 samples = 3 GiB).  The next nfb_render_backward on the same
 * handle consumes that state; weights must not be re-loaded in between.
 * Memory: when the records of the whole call would exceed the budget (environment NFB_TRAIN_MEM_MB, default 60 % of the free
 * device memory) — e.g. a full frame rendered with gradients enabled — the forward only renders (evaluation kernel) and the
 * backward re-runs the training forward chunk by chunk inside the budget: same gradients, one extra forward; the caller must
 * then keep the forward's input buffers alive until the backward, and explicit rays are required.
 * NFB_PREC_EXACT_GRAD: each tile record is 2 MiB — the first MiB exactly as in NFB_PREC_EXACT, the second the lo parts
 * lo = fp16(x - float(hi)) of every image (activations, encodings and the backward's gradients) at the same offsets
 * (nfb_layout.h kRecLo) — so records take twice the memory (2048 rays at 64+64 samples: 6 GiB), the memory budget above covers
 * half as many rays per chunk, and the backward moves about twice the record bytes. */
int nfb_render_forward_train(NfbHandle* h, const NfbRays* rays, const NfbSampling* sampling,
                             const NfbNoise* noise /* nullable */, const NfbOutputs* out, void* stream);

/* dL/d(outputs) of the 7-tuple; any member may be NULL (= zero).  All device pointers, shapes as NfbOutputs. */
typedef struct {
  const float* rgb_coarse;
  const float* disp_coarse;
  const float* acc_coarse;
  const float* rgb_fine;
  const float* disp_fine;
  const float* acc_fine;
  const float* w_last;
} NfbOutGrads;

/* Backward of the last nfb_render_forward_train: compositing backward -> tcgen05 dX chain -> tcgen05 weight-gradient GEMMs
 * -> gradients in the reference's parameter layout.  `params_*` are the 26 FP32 parameter pointers given to
 * nfb_load_weights; `grads_*` receive dL/dparam with the same shapes (entries 22, 23 = layers_dir.3.*, unused by the
 * forward, models.py:257: may be NULL and are never written).  `grad_latent` [32] receives dL/d latent_code (NULL: skipped);
 * the sample depths carry no gradient (z_samples.detach(), train_utils.py:124).  Gradients are OVERWRITTEN, not accumulated.
 * params_fine / grads_fine may be NULL when the forward had num_fine == 0. */
int nfb_render_backward(NfbHandle* h, const NfbOutGrads* out_grads, const float* const params_coarse[26],
                        const float* const params_fine[26], float* const grads_coarse[26], float* const grads_fine[26],
                        float* grad_latent, void* stream);

/* ---- Training-step tail: loss, optimizer, re-pack (replaces train_transformed_rays.py:355-400 for callers that adopt it;
 * the drop-in Python surface keeps working with torch.nn.functional.mse_loss + torch.optim.Adam) ----
 *
 * nfb_loss_mse_grad: d/d rgb of mse(rgb_coarse, target) + mse(rgb_fine, target) (train_transformed_rays.py:355-362, 382), the
 * means taken over n_total * 3 elements — n_total is the GLOBAL batch size when the n_rays of this call are one shard of it, so
 * that a SUM all-reduce of the parameter gradients gives the single-process gradient.  Writes grad_rgb_* [n_rays,3] (feed them
 * to nfb_render_backward) and ADDS this shard's share of the two loss values to loss[0], loss[1] (zero them first).  1 launch. */
int nfb_loss_mse_grad(NfbHandle* h, const float* rgb_coarse, const float* rgb_fine /* nullable */, const float* target,
                      int n_rays, long long n_total, float* grad_rgb_coarse, float* grad_rgb_fine, float* loss, void* stream);

/* torch.optim.Adam (betas, eps as given; no weight decay / amsgrad; YAML optimizer block) over ONE flat FP32 bucket of n
 * floats — the caller lays out both networks' parameters and the latent-code table in it and hands views of it to
 * nfb_render_backward as gradient targets, so neither a gradient copy nor a torch.cat precedes an all-reduce.  In place:
 * params, exp_avg, exp_avg_sq are updated, grads are multiplied by grad_scale before use and ZEROED afterwards
 * (optimizer.zero_grad()).  The latent-code regulariser 10 * 0.0005 * ||latent||_2 (train_transformed_rays.py:369-372, 386) is
 * applied here: reg_weight * l / ||l|| is added to the gradient of the 32 floats at reg_offset (reg_offset < 0: none).
 * `step` counts from 1; `lr` is this step's learning rate (the caller evaluates the schedule of :393-399).  1 launch. */
typedef struct {
  float lr, beta1, beta2, eps;
  int32_t step;
  float grad_scale;
  long long reg_offset;
  float reg_weight;
} NfbAdam;
int nfb_adam_step(NfbHandle* h, float* params, float* grads, float* exp_avg, float* exp_avg_sq, long long n, const NfbAdam* hp,
                  void* stream);

/* nfb_adam_step with its per-step scalars in DEVICE memory, so that a whole training iteration can be captured once in a CUDA graph
 * and replayed: `dev_state` points to an NfbAdamDev on the device.  Each call first advances `step` and evaluates the reference's
 * learning-rate schedule lr0 * decay_factor ^ ((i - 1) / decay_steps) for loop index i = step - 1 >= 1 (train_transformed_rays.py:393-399)
 * and the bias corrections on the device (1 thread, float64), then runs the Adam kernel.  The regularised row is
 * table_offset + 32 * row[0] (row = device pointer to the current latent index; table_offset < 0: no regulariser).  2 launches. */
typedef struct {
  int32_t step, pad;               /* in/out: steps taken so far (start at 0) */
  float lr0, decay_factor, decay_steps, beta1, beta2, eps, grad_scale, reg_weight;
  long long table_offset;
  const long long* row;
  float lr_over_bc1, sqrt_bc2;     /* out: this step's scalars (written by the prepare kernel) */
  long long reg_offset;            /* out */
} NfbAdamDev;
int nfb_adam_step_dev(NfbHandle* h, float* params, float* grads, float* exp_avg, float* exp_avg_sq, long long n, NfbAdamDev* dev_state,
                      void* stream);

/* nfb_load_weights for both networks at once (params_fine may be NULL), two launches (FP64 fold, pack): the re-pack after an
 * optimizer step. */
int nfb_repack(NfbHandle* h, const float* const params_coarse[26], const float* const params_fine[26], void* stream);

/* ---- The steps either side of the path (SURVEY.md 8f ranks 3, 4) ----
 *
 * nfb_frame_products: the 8-bit images eval_transformed_rays.py writes per rendered frame, from the path's outputs still on the
 * device: rgb_u8 = cast_to_image(rgb) (:184-192), normals_u8 [(H-1),(W-1),3] = torch_normal_map(disparity, intrinsics, w_last,
 * clean=True) (:84-119, called at :469 with disp_fine and weights_fine[:, -1]), disparity_u8 = cast_to_disparity_image (:195-198).
 * Any output (and w_last) may be NULL.  The bytes equal the reference functions' (same FP32 operation order).  torch's two back
 * ends round torch_normal_map differently in two places: CUDA turns ".../ fx" (division by a host scalar) into a multiplication by
 * the FP32 reciprocal and sums the normal's squared components as (x2 + z2) + y2; the CPU divides and sums (x2 + y2) + z2.  The
 * default follows the CUDA back end — what the eval script computes on a GPU; NFB_PRODUCTS_LIKE_TORCH_CPU follows the CPU back
 * end (the two differ by one level in ~2e-4 of the bytes).  Square frames only for the normal map (the reference's expression
 * does not broadcast otherwise).  1 launch (+1 for disparity_u8). */
enum { NFB_PRODUCTS_LIKE_TORCH_CPU = 1 };
int nfb_frame_products(NfbHandle* h, const float* rgb /* [H,W,3] */, const float* disparity /* [H,W] */,
                       const float* w_last /* [H,W] or NULL */, const double intrinsics[4], int height, int width, uint8_t* rgb_u8,
                       uint8_t* normals_u8, uint8_t* disparity_u8, int flags, void* stream);

/* Importance map of one training image (train_transformed_rays.py:230-239): probs[bbox[0]:bbox[1], bbox[2]:bbox[3]] = p, 1 - p
 * elsewhere, normalised; q_out / q_in are the two float64 values of the normalised map exactly as numpy produced them. */
typedef struct {
  int32_t height, width;
  int32_t bbox[4];
  double q_out, q_in;
} NfbRayMap;
/* Optional gathers of nfb_sample_rays (train_transformed_rays.py:323-331); every member may be NULL / unused.  Pixel of flat
 * index k: (row, col) = (k % height, k / height) — the reference's transposed-meshgrid indexing. */
typedef struct {
  float pose[12];            /* camera-to-world 3x4 of the frame: rays as get_ray_bundle would give them */
  double intrinsics[4];
  const float* image;        /* [H,W,3] device */
  const float* background;   /* [H,W,3] device */
  float* ray_origins;        /* [size,3] out */
  float* ray_directions;     /* [size,3] out */
  float* target;             /* [size,3] out */
  float* background_out;     /* [size,3] out */
  int32_t* pixel_rc;         /* [size,2] out */
} NfbRayGather;
/* np.random.choice(H * W, size, replace=False, p=map.reshape(-1)) (:319-321) on the device, bit-identical indices for the same
 * uniform draws: `draws` (device, float64 in [0,1)) is consumed exactly like RandomState.rand inside choice — round r reads
 * (size - n_found) values.  state (device int32[3] = n_found, rounds run, draws consumed; zero it to start) lets a caller that must
 * stay in lock-step with a host RNG run one round per call.  indices [size] receives the selection in numpy's order; size <= 2048.
 * 1 launch (one thread block; the float64 cumulative sum is evaluated exactly without being materialised, csrc/nfb_sampler.h). */
int nfb_sample_rays(NfbHandle* h, const NfbRayMap* map, const double* draws, int size, int max_rounds, long long* indices,
                    int32_t* state, const NfbRayGather* gather /* nullable */, void* stream);
/* Host-only test hook of the same arithmetic: out[i] = np.cumsum(p)[ks[i]] (ks[i] == -1: the last entry) for the map with the
 * ascending flat indices zeroed_sorted set to zero.  No CUDA call. */
int nfb_host_map_cdf(const NfbRayMap* map, const long long* zeroed_sorted, int n_zero, const long long* ks, int n, double* out);

/* Test hook: device pointers of the training state (valid until the next forward_train on the handle). */
typedef struct {
  const uint8_t* records;      /* n_tiles records of record_bytes (layout: nfb_layout.h kRec*; 2 MiB with the lo MiB at kRecLo
                                  after an NFB_PREC_EXACT_GRAD forward) */
  long long n_tiles;
  int32_t record_bytes;
  const float* d_raw;          /* [n_tiles][128][4] dL/d(rgb_raw, sigma_raw), unscaled */
  const float* acc_coarse;     /* acc_floats accumulators in the kernel's folded parametrisation (kAcc*) */
  const float* acc_fine;
  int32_t acc_floats;
  const float* scale;          /* [0] loss scale, [1] its inverse */
  const float *z_coarse, *raw_coarse, *z_fine, *raw_fine;
  int32_t tiles_coarse, tiles_fine, rays_per_unit;
} NfbTrainDebug;
int nfb_train_debug(NfbHandle* h, NfbTrainDebug* out);

/* End-to-end convenience for callers with HOST buffers (bench.py's e2e leg, C/C++ users): copies
 * expression/latent/background to the device, renders image rows [row_begin,row_begin+rows) of a
 * height x width frame with in-kernel ray generation, and copies the outputs back.  Host pointers
 * should be pinned for full copy speed.  Output layout: out_host = rgb_c[n,3] | disp_c[n] | acc_c[n] |
 * rgb_f[n,3] | disp_f[n] | acc_f[n] | w_last[n], n = rows*width, 11*n floats.  Synchronises `stream`. */
int nfb_render_frame_host(NfbHandle* h, const float pose[12], const double intrinsics[4],
                          int height, int width, int row_begin, int rows, float near_, float far_,
                          const float* expression_host, const float* latent_host,
                          const float* background_host /* [rows*width,3] or NULL */,
                          const NfbSampling* sampling, float* out_host, void* stream);

/* Test hook, host only (no CUDA call): the compile-time schedules the kernels execute.  which: 0 = one-tile render program,
 * 1 = two-tile render program (word 4 = half-step group), 2 = backward chain program (each: idesc, TMEM columns, flags,
 * (stream offset / 16) | rows << 20), 3 = weight-gradient jobs (a_off, a_rows, a_half, b_off, b_rows, bias_layer, out_off,
 * out_ld, out_row0, group), 4 = the CTA split of the weight-gradient launch (in/out: out[0..2] = SMs, tiles of network 0, tiles of
 * network 1 -> parts of network 0, parts of network 1, job groups per part), 5 = exact-gradient chain program (one entry per hi or
 * lo load: the entry of 2 with the stream_bwd_x3 offset, part, lo A column, shared-memory bytes, slot bytes, slots, operand buffers),
 * 6 = exact-gradient weight-gradient stages per job (stage offsets of A hi, B hi, A lo, B lo, stage bytes, stages, bytes per tile,
 * bytes per tile of the FP16 kernel, shared-memory bytes, lo record offset), 1000 + 100 n_iter + 10 Tc + Tf = the pipelined render kernel's job sequence for a CTA with n_iter units of work and
 * Tc / Tf tile pairs per pass (unit iteration, pass, tile, then the kernel's shared-memory bytes and row limits).  index < 0: returns the number of entries; otherwise fills out[0..] (out_words >= 10) and returns
 * the number of words written, or -1. */
int nfb_debug_schedule(int which, int index, uint32_t* out, int out_words);

/* Number of kernel launches issued by this handle so far (all kernels of this library). */
int nfb_launch_count(NfbHandle* h, long long* out);

/* Host helper: out[i] = torch.linspace(0, 1, n)[i] bit-for-bit (ATen's CPU kernel: step = 1/(n-1) in
 * FP32; first half start + i*step, second half end - (n-1-i)*step).  Used for t_coarse / u_fine when the
 * caller passes NULL.  No CUDA involved. */
int nfb_host_linspace(float* out, int n);

#ifdef __cplusplus
}
#endif
#endif /* NFB_H_ */
