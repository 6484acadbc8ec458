// nfb_api.cu — the C ABI declared in include/nfb.h: handle management, argument validation, and
// translation of the public structs into kernel launches.  No torch, no exceptions across the boundary.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/nfb.h"
#include "nfb_internal.h"
#include "nfb_layout.h"

namespace {
thread_local std::string g_last_cuda_error;

int cuda_fail(cudaError_t e, const char* where) {
  g_last_cuda_error = std::string(where) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
  return NFB_ERR_CUDA;
}
#define NFB_CUDA(call)                                   \
  do {                                                   \
    cudaError_t e__ = (call);                            \
    if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
  } while (0)

template <class T>
cudaError_t dev_alloc(T** p, size_t n) { return cudaMalloc(reinterpret_cast<void**>(p), n * sizeof(T)); }
}  // namespace

struct NfbHandle {
  int device = 0;
  int num_sms = 0;
  nfb::NetBuffers net[2];
  bool frame_set = false;
  bool use_render2 = true;
  bool use_render3 = true;
  long long launches = 0;
  // cached torch.linspace(0,1,n) tables on the device
  float* lin_c = nullptr; int lin_c_n = 0;
  float* lin_f = nullptr; int lin_f_n = 0;
  // staging for nfb_render_frame_host
  float *d_expr = nullptr, *d_latent = nullptr, *d_bg = nullptr, *d_out = nullptr;
  size_t bg_cap = 0, out_cap = 0;
  // training state: what nfb_render_forward_train saved for nfb_render_backward (grow-only buffers)
  struct Train {
    uint8_t* rec = nullptr; size_t rec_tiles = 0;       // per-tile activation records (nfb_layout.h kRec*), rec_tiles = bytes
    float* draw = nullptr; size_t draw_tiles = 0;       // [tiles][128][4]
    float *z_c = nullptr, *raw_c = nullptr, *z_f = nullptr, *raw_f = nullptr, *dnorm = nullptr;
    size_t cap_zc = 0, cap_rawc = 0, cap_zf = 0, cap_rawf = 0, cap_dn = 0;
    float* acc[2] = {nullptr, nullptr};                 // kAccFloats each
    float* scal = nullptr;                              // [0] scale, [1] 1/scale, [2] max |d raw| (bits)
    float* cond = nullptr;                              // [108] conditioning vector of the frame the forward rendered
    int n_rays = 0, nc = 0, nf = 0, rays_per_unit = 0, tiles_c = 0, tiles_f = 0, n_units = 0, has_bg = 0, white_bkgd = 0;
    bool valid = false;
    bool exact_grad = false;     // NFB_PREC_EXACT_GRAD: 2 MiB hi+lo records, exact chain and weight-gradient kernels
    // chunked mode (the records of the whole call would exceed the memory budget): the forward only produced the outputs; the
    // backward re-runs the training forward chunk by chunk from the saved launch parameters (the caller keeps the inputs alive)
    bool chunked = false;
    nfb::RenderParams full;      // the forward call's parameters (pointers into caller memory)
    int chunk_rays = 0, precision = 0;
    float* scratch_out = nullptr; size_t scratch_cap = 0;   // [11 * chunk_rays] outputs of the re-run forwards (discarded)
  } tr;
  size_t train_budget = 0;       // bytes the per-tile records of one launch may take (0: not decided yet)
  float* cond = nullptr;  // [108] = [expression / 3 ; latent] of the current frame
  // scratch of the steps either side of the path
  uint32_t* minmax = nullptr;                           // disparity-image min / max keys
  nfb::smp::Run* smp_runs = nullptr; nfb::smp::Seg* smp_segs = nullptr; int* smp_first = nullptr; long long smp_first_n = 0;
};

namespace {
template <class T>
int ensure_cap(T** p, size_t* cap, size_t n) {
  if (*cap >= n && *p) return NFB_OK;
  if (*p) NFB_CUDA(cudaFree(*p));
  *p = nullptr;
  *cap = 0;
  NFB_CUDA(cudaMalloc(reinterpret_cast<void**>(p), n * sizeof(T)));
  *cap = n;
  return NFB_OK;
}
}  // namespace

extern "C" {

int nfb_version(void) { return NFB_VERSION; }

const char* nfb_strerror(int status) {
  switch (status) {
    case NFB_OK: return "ok";
    case NFB_ERR_INVALID: return "invalid argument";
    case NFB_ERR_UNSUPPORTED: return "configuration not supported by the sm_100a render kernel";
    case NFB_ERR_CUDA: return "CUDA runtime error (see nfb_last_cuda_error)";
    case NFB_ERR_STATE: return "weights or per-frame conditioning not set";
    case NFB_ERR_ARCH: return "device is not compute capability 10.x (sm_100a code only)";
    default: return "unknown status";
  }
}

const char* nfb_last_cuda_error(void) { return g_last_cuda_error.c_str(); }

int nfb_host_linspace(float* out, int n) {
  if (!out || n < 1) return NFB_ERR_INVALID;
  if (n == 1) { out[0] = 0.f; return NFB_OK; }
  // ATen's CPU linspace: symmetric evaluation about the midpoint, all in FP32.
  const float start = 0.f, end = 1.f;
  const float step = (end - start) / static_cast<float>(n - 1);
  const int halfway = n / 2;
  for (int i = 0; i < n; ++i) out[i] = (i < halfway) ? start + step * static_cast<float>(i) : end - step * static_cast<float>(n - i - 1);
  return NFB_OK;
}

static int create_impl(NfbHandle* h, const cudaDeviceProp& prop) {
  h->num_sms = prop.multiProcessorCount;
  for (int n = 0; n < 2; ++n) {
    nfb::NetBuffers& nb = h->net[n];
    NFB_CUDA(dev_alloc(&nb.stream_x1, nfb::kStreamBytesX1));
    NFB_CUDA(dev_alloc(&nb.stream_x3, nfb::kStreamBytesX3));
    NFB_CUDA(dev_alloc(&nb.w6, 144 * 256));
    NFB_CUDA(dev_alloc(&nb.b6, 144));
    NFB_CUDA(dev_alloc(&nb.bias_static, nfb::kBiasFloats));
    NFB_CUDA(dev_alloc(&nb.bias_frame, nfb::kBiasFloats));
    NFB_CUDA(dev_alloc(&nb.w0c, 256 * nfb::kDimCond));
    NFB_CUDA(dev_alloc(&nb.w3c, 256 * nfb::kDimCond));
    NFB_CUDA(dev_alloc(&nb.wd0b_t, nfb::kDimDir * 128));
    NFB_CUDA(dev_alloc(&nb.stream_bwd, nfb::kBwdStreamBytes));
    NFB_CUDA(dev_alloc(&nb.stream_bwd_x3, nfb::kBwdStreamBytesX3));
    NFB_CUDA(dev_alloc(&h->tr.acc[n], nfb::kAccFloats));
  }
  NFB_CUDA(dev_alloc(&h->tr.scal, 4));
  NFB_CUDA(dev_alloc(&h->tr.cond, nfb::kDimCond));
  NFB_CUDA(dev_alloc(&h->cond, nfb::kDimCond));
  NFB_CUDA(nfb::train_kernels_setup());
  NFB_CUDA(dev_alloc(&h->d_expr, nfb::kDimExpr));
  NFB_CUDA(dev_alloc(&h->d_latent, nfb::kDimLatent));
  NFB_CUDA(nfb::render_kernel_setup());
  NFB_CUDA(nfb::render2_kernel_setup());
  NFB_CUDA(nfb::render3_kernel_setup());
  {  // NFB_KERNEL=v4 forces the one-tile-in-flight kernel everywhere (default: the two-tile kernel where it applies)
    const char* k = std::getenv("NFB_KERNEL");
    h->use_render2 = !(k && std::strcmp(k, "v4") == 0);
    h->use_render3 = h->use_render2 && !(k && std::strcmp(k, "v6") == 0);  // NFB_KERNEL=v6: two tiles in flight, passes not pipelined
  }
  return NFB_OK;
}


int nfb_create(const NfbModelDims* dims, int device, NfbHandle** out) {
  if (!dims || !out) return NFB_ERR_INVALID;
  if (dims->num_encoding_fn_xyz != 10 || dims->num_encoding_fn_dir != 4 || dims->include_input_xyz != 1 ||
      dims->include_input_dir != 0 || dims->dim_expression != nfb::kDimExpr || dims->dim_latent != nfb::kDimLatent)
    return NFB_ERR_UNSUPPORTED;
  NFB_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  NFB_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return NFB_ERR_ARCH;
  NfbHandle* h = new (std::nothrow) NfbHandle();
  if (!h) return NFB_ERR_INVALID;
  h->device = device;
  const int rc = create_impl(h, prop);
  if (rc != NFB_OK) {  // free whatever was allocated before the failure
    nfb_destroy(h);
    return rc;
  }
  *out = h;
  return NFB_OK;
}

int nfb_destroy(NfbHandle* h) {
  if (!h) return NFB_ERR_INVALID;
  cudaSetDevice(h->device);
  for (int n = 0; n < 2; ++n) {
    nfb::NetBuffers& nb = h->net[n];
    cudaFree(nb.stream_x1); cudaFree(nb.stream_x3); cudaFree(nb.w6); cudaFree(nb.b6); cudaFree(nb.bias_static);
    cudaFree(nb.bias_frame); cudaFree(nb.w0c); cudaFree(nb.w3c); cudaFree(nb.wd0b_t); cudaFree(nb.stream_bwd);
    cudaFree(nb.stream_bwd_x3);
    cudaFree(h->tr.acc[n]);
  }
  cudaFree(h->tr.rec); cudaFree(h->tr.draw); cudaFree(h->tr.z_c); cudaFree(h->tr.raw_c); cudaFree(h->tr.z_f); cudaFree(h->tr.raw_f);
  cudaFree(h->tr.dnorm); cudaFree(h->tr.scal); cudaFree(h->tr.cond); cudaFree(h->tr.scratch_out); cudaFree(h->cond);
  cudaFree(h->minmax); cudaFree(h->smp_runs); cudaFree(h->smp_segs); cudaFree(h->smp_first);
  cudaFree(h->lin_c); cudaFree(h->lin_f); cudaFree(h->d_expr); cudaFree(h->d_latent); cudaFree(h->d_bg); cudaFree(h->d_out);
  delete h;
  return NFB_OK;
}

int nfb_load_weights(NfbHandle* h, int which, const float* const params[26], void* stream) {
  if (!h || !params || (which != NFB_NET_COARSE && which != NFB_NET_FINE)) return NFB_ERR_INVALID;
  for (int i = 0; i < 26; ++i)
    if (!params[i]) return NFB_ERR_INVALID;
  NFB_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  nfb::NetBuffers& nb = h->net[which];
  nfb::NetBuffers* const nbs[2] = {&nb, nullptr};
  const float* const* const ps[2] = {params, nullptr};
  NFB_CUDA(nfb::launch_repack(nbs, ps, 1, st, &h->launches));  // forward streams, transposed backward stream, bias / column blocks
  nb.loaded = true;
  h->frame_set = false;  // folded biases are stale
  return NFB_OK;
}

int nfb_repack(NfbHandle* h, const float* const params_coarse[26], const float* const params_fine[26], void* stream) {
  if (!h || !params_coarse) return NFB_ERR_INVALID;
  for (int i = 0; i < 26; ++i)
    if (!params_coarse[i] || (params_fine && !params_fine[i])) return NFB_ERR_INVALID;
  NFB_CUDA(cudaSetDevice(h->device));
  nfb::NetBuffers* const nbs[2] = {&h->net[0], &h->net[1]};
  const float* const* const ps[2] = {params_coarse, params_fine};
  NFB_CUDA(nfb::launch_repack(nbs, ps, params_fine ? 2 : 1, static_cast<cudaStream_t>(stream), &h->launches));
  h->net[0].loaded = true;
  if (params_fine) h->net[1].loaded = true;
  h->frame_set = false;  // folded biases are stale
  return NFB_OK;
}

int nfb_loss_mse_grad(NfbHandle* h, const float* rgb_coarse, const float* rgb_fine, const float* target, int n_rays,
                      long long n_total, float* grad_rgb_coarse, float* grad_rgb_fine, float* loss, void* stream) {
  if (!h || !rgb_coarse || !target || !grad_rgb_coarse || !loss || n_rays < 0 || n_total < n_rays || n_total <= 0) return NFB_ERR_INVALID;
  if (rgb_fine && !grad_rgb_fine) return NFB_ERR_INVALID;
  NFB_CUDA(cudaSetDevice(h->device));
  NFB_CUDA(nfb::launch_loss_grad(rgb_coarse, rgb_fine, target, n_rays, n_total, grad_rgb_coarse, grad_rgb_fine, loss,
                                 static_cast<cudaStream_t>(stream), &h->launches));
  return NFB_OK;
}

int nfb_adam_step(NfbHandle* h, float* params, float* grads, float* exp_avg, float* exp_avg_sq, long long n, const NfbAdam* hp,
                  void* stream) {
  if (!h || !params || !grads || !exp_avg || !exp_avg_sq || !hp || n <= 0 || hp->step < 1) return NFB_ERR_INVALID;
  // the regularised row must not straddle two 256-float chunks (one thread block each): its norm is taken per block
  if (hp->reg_offset >= 0 && (hp->reg_offset + nfb::kDimLatent > n || hp->reg_offset % nfb::kDimLatent != 0)) return NFB_ERR_INVALID;
  NFB_CUDA(cudaSetDevice(h->device));
  NFB_CUDA(nfb::launch_adam(params, grads, exp_avg, exp_avg_sq, n, hp->lr, hp->beta1, hp->beta2, hp->eps, hp->step, hp->grad_scale,
                            hp->reg_offset, hp->reg_weight, static_cast<cudaStream_t>(stream), &h->launches));
  return NFB_OK;
}

int nfb_adam_step_dev(NfbHandle* h, float* params, float* grads, float* exp_avg, float* exp_avg_sq, long long n, NfbAdamDev* dev_state,
                      void* stream) {
  if (!h || !params || !grads || !exp_avg || !exp_avg_sq || !dev_state || n <= 0) return NFB_ERR_INVALID;
  NFB_CUDA(cudaSetDevice(h->device));
  NFB_CUDA(nfb::launch_adam_dev(params, grads, exp_avg, exp_avg_sq, n, dev_state, static_cast<cudaStream_t>(stream), &h->launches));
  return NFB_OK;
}

int nfb_set_frame(NfbHandle* h, const float* expression, const float* latent, void* stream) {
  if (!h || !expression || !latent) return NFB_ERR_INVALID;
  if (!h->net[0].loaded) return NFB_ERR_STATE;
  NFB_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  nfb::NetBuffers* const nbs[2] = {&h->net[0], &h->net[1]};
  NFB_CUDA(nfb::launch_frame_fold(nbs, h->net[1].loaded ? 2 : 1, expression, latent, h->cond, st, &h->launches));
  h->frame_set = true;
  return NFB_OK;
}

static int ensure_linspace(float** buf, int* cached_n, int n, cudaStream_t st) {
  if (*cached_n == n && *buf) return NFB_OK;
  std::vector<float> host(n);
  nfb_host_linspace(host.data(), n);
  if (*buf) NFB_CUDA(cudaFree(*buf));
  *buf = nullptr;
  *cached_n = 0;
  NFB_CUDA(dev_alloc(buf, (size_t)n));
  // pageable source: the runtime stages it before returning, so `host` may die afterwards
  NFB_CUDA(cudaMemcpyAsync(*buf, host.data(), n * sizeof(float), cudaMemcpyHostToDevice, st));
  *cached_n = n;
  return NFB_OK;
}

// Memory the per-tile activation records of ONE training launch may take: NFB_TRAIN_MEM_MB, else 60 % of the device memory that
// is free when first asked (at least 1 GiB).  A call that needs more is processed in ray chunks (see NfbHandle::Train::chunked).
static size_t train_budget(NfbHandle* h) {
  if (const char* e = std::getenv("NFB_TRAIN_MEM_MB")) {  // read on every call: tests switch it within one process
    const size_t mb = (size_t)std::strtoull(e, nullptr, 10);
    if (mb) return mb << 20;
  }
  if (h->train_budget) return h->train_budget;
  size_t budget = 0;
  {
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) budget = free_b / 10 * 6;
  }
  if (budget < ((size_t)1 << 30)) budget = (size_t)1 << 30;
  return h->train_budget = budget;
}

// (Re)size the buffers a training launch over n rays / `tiles` tiles writes (records of tr.exact_grad's size).
static int ensure_train_buffers(NfbHandle::Train& tr, size_t n, size_t tiles, int nc, int nf) {
  int rc;
  if ((rc = ensure_cap(&tr.rec, &tr.rec_tiles, tiles * (size_t)nfb::rec_stride(tr.exact_grad)))) return rc;
  if ((rc = ensure_cap(&tr.draw, &tr.draw_tiles, tiles * 512))) return rc;
  if ((rc = ensure_cap(&tr.z_c, &tr.cap_zc, n * nc))) return rc;
  if ((rc = ensure_cap(&tr.raw_c, &tr.cap_rawc, n * nc * 4))) return rc;
  if ((rc = ensure_cap(&tr.dnorm, &tr.cap_dn, n))) return rc;
  if (nf > 0) {
    if ((rc = ensure_cap(&tr.z_f, &tr.cap_zf, n * (nc + nf)))) return rc;
    if ((rc = ensure_cap(&tr.raw_f, &tr.cap_rawf, n * (nc + nf) * 4))) return rc;
  }
  return NFB_OK;
}

static int render_impl(NfbHandle* h, const NfbRays* rays, const NfbSampling* sm, const NfbNoise* noise, const NfbOutputs* out,
                       const NfbDebug* dbg, void* stream, bool train) {
  if (!h || !rays || !sm || !out) return NFB_ERR_INVALID;
  if (rays->n_rays < 0) return NFB_ERR_INVALID;
  if ((rays->o == nullptr) != (rays->d == nullptr)) return NFB_ERR_INVALID;
  if (!rays->o && (rays->width <= 0 || rays->height <= 0)) return NFB_ERR_INVALID;
  const int nc = sm->num_coarse, nf = sm->num_fine;
  if (nc < 3 || nf < 0 || nc + nf > 512) return NFB_ERR_UNSUPPORTED;
  if (sm->lindisp) return NFB_ERR_UNSUPPORTED;
  if (sm->precision != NFB_PREC_FAST && sm->precision != NFB_PREC_EXACT && sm->precision != NFB_PREC_EXACT_GRAD) return NFB_ERR_INVALID;
  if (!h->net[0].loaded || (nf > 0 && !h->net[1].loaded) || !h->frame_set) return NFB_ERR_STATE;
  if (!out->rgb_coarse || !out->disp_coarse || !out->acc_coarse) return NFB_ERR_INVALID;
  if (nf > 0 && (!out->rgb_fine || !out->disp_fine || !out->acc_fine)) return NFB_ERR_INVALID;
  if (sm->perturb && (!noise || !noise->t_rand || (nf > 0 && !noise->u))) return NFB_ERR_INVALID;
  if (sm->noise_std > 0.f && (!noise || !noise->sigma_noise_c || (nf > 0 && !noise->sigma_noise_f))) return NFB_ERR_INVALID;
  if (rays->n_rays == 0) return NFB_OK;
  NFB_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);

  nfb::RenderParams p;
  std::memset(&p, 0, sizeof(p));
  p.o = rays->o; p.d = rays->d; p.n_rays = rays->n_rays;
  for (int i = 0; i < 12; ++i) p.pose[i] = rays->pose[i];
  p.fx = static_cast<float>(rays->intrinsics[0]);
  p.fy = static_cast<float>(rays->intrinsics[1]);
  p.wcx = static_cast<float>(static_cast<double>(rays->width) * rays->intrinsics[2]);
  p.hcy = static_cast<float>(static_cast<double>(rays->height) * rays->intrinsics[3]);
  p.width = rays->width > 0 ? rays->width : 1;
  p.row_begin = rays->row_begin;
  p.near_ = rays->near_; p.far_ = rays->far_;
  p.dir_z = rays->dir_z; p.bg = rays->background;
  p.nc = nc; p.nf = nf; p.s_fine = nc + nf;
  p.rays_per_unit = (2 * (nc + nf) <= 512) ? 2 : 1;
  p.tiles_c = (p.rays_per_unit * nc + 127) / 128;
  p.tiles_f = nf > 0 ? (p.rays_per_unit * (nc + nf) + 127) / 128 : 0;
  p.n_units = (rays->n_rays + p.rays_per_unit - 1) / p.rays_per_unit;
  p.perturb = sm->perturb ? 1 : 0;
  p.noise_std = sm->noise_std;
  p.white_bkgd = sm->white_background ? 1 : 0;
  if (sm->t_coarse) p.t_coarse = sm->t_coarse;
  else {
    int rc = ensure_linspace(&h->lin_c, &h->lin_c_n, nc, st);
    if (rc) return rc;
    p.t_coarse = h->lin_c;
  }
  if (nf > 0) {
    if (sm->u_fine) p.u_fine = sm->u_fine;
    else {
      int rc = ensure_linspace(&h->lin_f, &h->lin_f_n, nf, st);
      if (rc) return rc;
      p.u_fine = h->lin_f;
    }
  }
  if (noise) { p.t_rand = noise->t_rand; p.noise_c = noise->sigma_noise_c; p.u_rand = noise->u; p.noise_f = noise->sigma_noise_f; }
  const bool exact = sm->precision != NFB_PREC_FAST;  // NFB_PREC_EXACT_GRAD renders with the exact kernels too
  for (int n = 0; n < 2; ++n) {
    p.wstream[n] = exact ? h->net[n].stream_x3 : h->net[n].stream_x1;
    p.bias[n] = h->net[n].bias_frame;
    p.wd0b_t[n] = h->net[n].wd0b_t;
  }
  if (nf == 0) { p.wstream[1] = p.wstream[0]; p.bias[1] = p.bias[0]; p.wd0b_t[1] = p.wd0b_t[0]; }
  p.rgb_c = out->rgb_coarse; p.disp_c = out->disp_coarse; p.acc_c = out->acc_coarse;
  p.rgb_f = out->rgb_fine; p.disp_f = out->disp_fine; p.acc_f = out->acc_fine; p.w_last = out->w_last;
  if (dbg) {
    p.dbg_z_c = dbg->z_coarse; p.dbg_raw_c = dbg->raw_coarse; p.dbg_z_f = dbg->z_fine; p.dbg_raw_f = dbg->raw_fine;
    p.dbg_act = dbg->act_dump; p.dbg_act_step = dbg->act_step; p.prof = dbg->prof;
  }
  if (train) {
    // Saved for nfb_render_backward: per-tile activation records, sample depths, (colour, ReLU input of sigma), |d|.
    NfbHandle::Train& tr = h->tr;
    tr.valid = false;
    tr.exact_grad = sm->precision == NFB_PREC_EXACT_GRAD;
    const size_t rec_bytes = (size_t)nfb::rec_stride(tr.exact_grad);
    const size_t n = (size_t)rays->n_rays, tiles_per_unit = (size_t)(p.tiles_c + p.tiles_f), tiles = (size_t)p.n_units * tiles_per_unit;
    int rc;
    tr.chunked = tiles * rec_bytes > train_budget(h);
    if (tr.chunked) {
      // e.g. a whole frame rendered with gradients enabled: 1.5-2 MiB of records per ray.  Keep the launch parameters, produce
      // the outputs with the evaluation kernel now, and let the backward re-run the training forward in chunks that fit.
      if (!rays->o) { g_last_cuda_error = "training forward over budget needs explicit rays (o, d)"; return NFB_ERR_UNSUPPORTED; }
      size_t units = train_budget(h) / rec_bytes / tiles_per_unit;
      units &= ~(size_t)1;  // whole two-tile units of work
      if (units < 2) units = 2;
      tr.chunk_rays = (int)(units * p.rays_per_unit);
      tr.full = p;
      tr.precision = tr.exact_grad ? 2 : (exact ? 1 : 0);
    } else if ((rc = ensure_train_buffers(tr, n, tiles, nc, nf))) return rc;
    // a later nfb_set_frame (e.g. a validation render before the backward) must not change what the backward differentiates
    NFB_CUDA(cudaMemcpyAsync(tr.cond, h->cond, nfb::kDimCond * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (!tr.chunked) {
      p.save_rec = tr.rec; p.save_dnorm = tr.dnorm; p.save_raw_c = tr.raw_c; p.save_raw_f = tr.raw_f;
      p.dbg_z_c = tr.z_c; p.dbg_z_f = tr.z_f;
    }
    tr.n_rays = rays->n_rays; tr.nc = nc; tr.nf = nf; tr.rays_per_unit = p.rays_per_unit; tr.tiles_c = p.tiles_c;
    tr.tiles_f = p.tiles_f; tr.n_units = p.n_units; tr.has_bg = rays->background != nullptr; tr.white_bkgd = p.white_bkgd;
  }
  // fast-mode evaluation runs a two-tiles-in-flight kernel; exact mode (hi+lo operands need twice the TMEM columns), the
  // training forward (only the one-tile kernel writes the activation records) and the layer probe run the one-tile kernel
  const bool saving = p.save_rec != nullptr;
  const bool two_tile = h->use_render2 && !exact && !p.dbg_act && !saving;
  const bool pipelined = two_tile && h->use_render3 && nfb::render3_supports(p);
  if (pipelined) NFB_CUDA(nfb::launch_render3(p, h->num_sms, st, &h->launches));
  else if (two_tile) NFB_CUDA(nfb::launch_render2(p, h->num_sms, st, &h->launches));
  else NFB_CUDA(nfb::launch_render(p, (saving && h->tr.exact_grad) ? 2 : (exact ? 1 : 0), h->num_sms, st, &h->launches));
  if (train) h->tr.valid = true;
  return NFB_OK;
}

int nfb_render_forward(NfbHandle* h, const NfbRays* rays, const NfbSampling* sm, const NfbNoise* noise, const NfbOutputs* out,
                       const NfbDebug* dbg, void* stream) {
  return render_impl(h, rays, sm, noise, out, dbg, stream, false);
}

int nfb_render_forward_train(NfbHandle* h, const NfbRays* rays, const NfbSampling* sm, const NfbNoise* noise,
                             const NfbOutputs* out, void* stream) {
  return render_impl(h, rays, sm, noise, out, nullptr, stream, true);
}

int nfb_render_backward(NfbHandle* h, const NfbOutGrads* og, const float* const params_coarse[26],
                        const float* const params_fine[26], float* const grads_coarse[26], float* const grads_fine[26],
                        float* grad_latent, void* stream) {
  if (!h || !og || !params_coarse || !grads_coarse) return NFB_ERR_INVALID;
  NfbHandle::Train& tr = h->tr;
  if (!tr.valid) return NFB_ERR_STATE;
  const bool fine = tr.nf > 0;
  if (fine && (!params_fine || !grads_fine)) return NFB_ERR_INVALID;
  for (int i = 0; i < 26; ++i) {
    if (!params_coarse[i] || (fine && !params_fine[i])) return NFB_ERR_INVALID;
    if (i != 22 && i != 23 && (!grads_coarse[i] || (fine && !grads_fine[i]))) return NFB_ERR_INVALID;
  }
  NFB_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  NFB_CUDA(cudaMemsetAsync(tr.acc[0], 0, nfb::kAccFloats * sizeof(float), st));
  NFB_CUDA(cudaMemsetAsync(tr.acc[1], 0, nfb::kAccFloats * sizeof(float), st));

  // compositing backward -> dX chain -> weight-gradient GEMMs for the rays [begin, begin + n) whose training state the buffers
  // hold; the FP32 accumulators tr.acc add up over chunks (each chunk has its own power-of-two loss scale, divided out again
  // before the accumulation)
  auto backward_rays = [&](int begin, int n, int n_units) -> int {
    const size_t tiles = (size_t)n_units * (tr.tiles_c + tr.tiles_f);
    NFB_CUDA(cudaMemsetAsync(tr.draw, 0, tiles * 512 * sizeof(float), st));
    NFB_CUDA(cudaMemsetAsync(tr.scal, 0, 4 * sizeof(float), st));
    nfb::CompBwdParams q;
    std::memset(&q, 0, sizeof(q));
    q.n_rays = n; q.nc = tr.nc; q.nf = tr.nf; q.s_fine = tr.nc + tr.nf; q.rays_per_unit = tr.rays_per_unit;
    q.tiles_c = tr.tiles_c; q.tiles_f = tr.tiles_f; q.has_bg = tr.has_bg; q.white_bkgd = tr.white_bkgd;
    q.z_c = tr.z_c; q.raw_c = tr.raw_c; q.z_f = tr.z_f; q.raw_f = tr.raw_f; q.dnorm = tr.dnorm;
    auto off3 = [&](const float* p) { return p ? p + 3 * (size_t)begin : nullptr; };
    auto off1 = [&](const float* p) { return p ? p + (size_t)begin : nullptr; };
    q.g_rgb[0] = off3(og->rgb_coarse); q.g_disp[0] = off1(og->disp_coarse); q.g_acc[0] = off1(og->acc_coarse);
    q.g_rgb[1] = off3(og->rgb_fine); q.g_disp[1] = off1(og->disp_fine); q.g_acc[1] = off1(og->acc_fine); q.g_wlast = off1(og->w_last);
    q.draw = tr.draw; q.acc[0] = tr.acc[0]; q.acc[1] = tr.acc[1];
    q.absmax = reinterpret_cast<unsigned int*>(tr.scal + 2);
    NFB_CUDA(nfb::launch_composite_bwd(q, tr.scal, st, &h->launches));

    nfb::ChainParams c;
    c.n_units = n_units; c.tiles_c = tr.tiles_c; c.tiles_f = tr.tiles_f;
    c.rec = tr.rec; c.draw = tr.draw; c.scal = tr.scal;
    const int fn = fine ? 1 : 0;
    c.wstream[0] = tr.exact_grad ? h->net[0].stream_bwd_x3 : h->net[0].stream_bwd;
    c.wstream[1] = tr.exact_grad ? h->net[fn].stream_bwd_x3 : h->net[fn].stream_bwd;
    NFB_CUDA(nfb::launch_chain(c, tr.exact_grad, h->num_sms, st, &h->launches));
    {
      nfb::DwParams d = {};
      d.rec = tr.rec; d.n_units = n_units; d.tpu = tr.tiles_c + tr.tiles_f;
      d.t_base[0] = 0; d.t_cnt[0] = tr.tiles_c;
      d.t_base[1] = tr.tiles_c; d.t_cnt[1] = fine ? tr.tiles_f : 0;
      d.acc[0] = tr.acc[0]; d.acc[1] = tr.acc[1]; d.scal = tr.scal;
      NFB_CUDA(nfb::launch_dw(d, tr.exact_grad, h->num_sms, st, &h->launches));  // both networks in one launch
    }
    return NFB_OK;
  };

  if (!tr.chunked) {
    int rc = backward_rays(0, tr.n_rays, tr.n_units);
    if (rc) return rc;
  } else {
    const int R = tr.rays_per_unit;
    for (int begin = 0; begin < tr.n_rays; begin += tr.chunk_rays) {
      const int n = tr.n_rays - begin < tr.chunk_rays ? tr.n_rays - begin : tr.chunk_rays;
      const int n_units = (n + R - 1) / R;
      const size_t tiles = (size_t)n_units * (tr.tiles_c + tr.tiles_f);
      int rc = ensure_train_buffers(tr, (size_t)n, tiles, tr.nc, tr.nf);
      if (rc) return rc;
      if (tr.scratch_cap < 11 * (size_t)tr.chunk_rays) {
        if (tr.scratch_out) NFB_CUDA(cudaFree(tr.scratch_out));
        tr.scratch_out = nullptr; tr.scratch_cap = 0;
        NFB_CUDA(dev_alloc(&tr.scratch_out, 11 * (size_t)tr.chunk_rays));
        tr.scratch_cap = 11 * (size_t)tr.chunk_rays;
      }
      // the training forward of this chunk: the saved launch with every per-ray pointer advanced to `begin`
      nfb::RenderParams p = tr.full;
      const size_t b = (size_t)begin;
      p.o += 3 * b; p.d += 3 * b; p.n_rays = n; p.n_units = n_units;
      if (p.dir_z) p.dir_z += b;
      if (p.bg) p.bg += 3 * b;
      if (p.t_rand) p.t_rand += b * tr.nc;
      if (p.noise_c) p.noise_c += b * tr.nc;
      if (p.u_rand) p.u_rand += b * tr.nf;
      if (p.noise_f) p.noise_f += b * (tr.nc + tr.nf);
      float* so = tr.scratch_out;
      const size_t cn = (size_t)tr.chunk_rays;
      p.rgb_c = so; p.disp_c = so + 3 * cn; p.acc_c = so + 4 * cn; p.rgb_f = so + 5 * cn; p.disp_f = so + 8 * cn; p.acc_f = so + 9 * cn;
      p.w_last = so + 10 * cn;
      p.save_rec = tr.rec; p.save_dnorm = tr.dnorm; p.save_raw_c = tr.raw_c; p.save_raw_f = tr.raw_f;
      p.dbg_z_c = tr.z_c; p.dbg_z_f = tr.z_f;
      NFB_CUDA(nfb::launch_render(p, tr.precision, h->num_sms, st, &h->launches));
      rc = backward_rays(begin, n, n_units);
      if (rc) return rc;
    }
  }
  NFB_CUDA(nfb::launch_finalize_all(params_coarse, grads_coarse, tr.acc[0], fine ? params_fine : nullptr, fine ? grads_fine : nullptr,
                                    tr.acc[1], tr.cond, grad_latent, st, &h->launches));
  return NFB_OK;
}

int nfb_train_debug(NfbHandle* h, NfbTrainDebug* out) {
  if (!h || !out) return NFB_ERR_INVALID;
  if (!h->tr.valid || h->tr.chunked) return NFB_ERR_STATE;  // chunked: the buffers only ever hold one chunk
  const NfbHandle::Train& tr = h->tr;
  out->records = tr.rec; out->n_tiles = (long long)tr.n_units * (tr.tiles_c + tr.tiles_f); out->record_bytes = (int32_t)nfb::rec_stride(tr.exact_grad);
  out->d_raw = tr.draw; out->acc_coarse = tr.acc[0]; out->acc_fine = tr.acc[1]; out->acc_floats = nfb::kAccFloats;
  out->scale = tr.scal; out->z_coarse = tr.z_c; out->raw_coarse = tr.raw_c; out->z_fine = tr.z_f; out->raw_fine = tr.raw_f;
  out->tiles_coarse = tr.tiles_c; out->tiles_fine = tr.tiles_f; out->rays_per_unit = tr.rays_per_unit;
  return NFB_OK;
}

int nfb_render_frame_host(NfbHandle* h, const float pose[12], const double intrinsics[4], int height, int width, int row_begin,
                          int rows, float near_, float far_, const float* expression_host, const float* latent_host,
                          const float* background_host, const NfbSampling* sm, float* out_host, void* stream) {
  if (!h || !pose || !intrinsics || !expression_host || !latent_host || !sm || !out_host) return NFB_ERR_INVALID;
  if (height <= 0 || width <= 0 || rows <= 0 || row_begin < 0 || row_begin + rows > height) return NFB_ERR_INVALID;
  if (sm->perturb || sm->noise_std > 0.f) return NFB_ERR_UNSUPPORTED;  // host path is the deterministic renderer
  NFB_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t n = (size_t)rows * width;
  if (h->out_cap < 11 * n) {
    if (h->d_out) NFB_CUDA(cudaFree(h->d_out));
    h->d_out = nullptr; h->out_cap = 0;
    NFB_CUDA(dev_alloc(&h->d_out, 11 * n));
    h->out_cap = 11 * n;
  }
  if (background_host && h->bg_cap < 3 * n) {
    if (h->d_bg) NFB_CUDA(cudaFree(h->d_bg));
    h->d_bg = nullptr; h->bg_cap = 0;
    NFB_CUDA(dev_alloc(&h->d_bg, 3 * n));
    h->bg_cap = 3 * n;
  }
  NFB_CUDA(cudaMemcpyAsync(h->d_expr, expression_host, nfb::kDimExpr * sizeof(float), cudaMemcpyHostToDevice, st));
  NFB_CUDA(cudaMemcpyAsync(h->d_latent, latent_host, nfb::kDimLatent * sizeof(float), cudaMemcpyHostToDevice, st));
  if (background_host) NFB_CUDA(cudaMemcpyAsync(h->d_bg, background_host, 3 * n * sizeof(float), cudaMemcpyHostToDevice, st));
  int rc = nfb_set_frame(h, h->d_expr, h->d_latent, stream);
  if (rc) return rc;
  NfbRays r;
  std::memset(&r, 0, sizeof(r));
  r.n_rays = (int)n;
  for (int i = 0; i < 12; ++i) r.pose[i] = pose[i];
  for (int i = 0; i < 4; ++i) r.intrinsics[i] = intrinsics[i];
  r.height = height; r.width = width; r.row_begin = row_begin;
  r.near_ = near_; r.far_ = far_;
  r.background = background_host ? h->d_bg : nullptr;
  NfbOutputs o;
  float* b = h->d_out;
  o.rgb_coarse = b; o.disp_coarse = b + 3 * n; o.acc_coarse = b + 4 * n;
  o.rgb_fine = b + 5 * n; o.disp_fine = b + 8 * n; o.acc_fine = b + 9 * n; o.w_last = b + 10 * n;
  rc = nfb_render_forward(h, &r, sm, nullptr, &o, nullptr, stream);
  if (rc) return rc;
  NFB_CUDA(cudaMemcpyAsync(out_host, h->d_out, 11 * n * sizeof(float), cudaMemcpyDeviceToHost, st));
  NFB_CUDA(cudaStreamSynchronize(st));
  return NFB_OK;
}

int nfb_frame_products(NfbHandle* h, const float* rgb, const float* disparity, const float* w_last, const double intrinsics[4], int height,
                       int width, uint8_t* rgb_u8, uint8_t* normals_u8, uint8_t* disparity_u8, int flags, void* stream) {
  if (!h || !intrinsics || height < 2 || width < 2) return NFB_ERR_INVALID;
  if ((rgb_u8 && !rgb) || ((normals_u8 || disparity_u8) && !disparity)) return NFB_ERR_INVALID;
  if (normals_u8 && height != width) return NFB_ERR_UNSUPPORTED;  // the reference's expression only broadcasts for square frames
  NFB_CUDA(cudaSetDevice(h->device));
  if (!h->minmax) NFB_CUDA(dev_alloc(&h->minmax, 2));
  NFB_CUDA(nfb::launch_frame_products(rgb, disparity, w_last, intrinsics, height, width, rgb_u8, normals_u8, disparity_u8, h->minmax,
                                      (flags & NFB_PRODUCTS_LIKE_TORCH_CPU) ? 1 : 0, static_cast<cudaStream_t>(stream), &h->launches));
  return NFB_OK;
}

int nfb_sample_rays(NfbHandle* h, const NfbRayMap* map, const double* draws, int size, int max_rounds, long long* indices, int32_t* state,
                    const NfbRayGather* g, void* stream) {
  if (!h || !map || !draws || !indices || !state || size < 1 || size > nfb::kSmpMax || max_rounds < 1) return NFB_ERR_INVALID;
  if (map->height < 1 || map->width < 1 || (long long)map->height * map->width < size) return NFB_ERR_INVALID;
  if (map->bbox[0] < 0 || map->bbox[1] > map->height || map->bbox[2] < 0 || map->bbox[3] > map->width) return NFB_ERR_INVALID;
  if (!(map->q_out > 0.0) || !(map->q_in > 0.0)) return NFB_ERR_INVALID;
  if (1 + 2 * (map->bbox[1] - map->bbox[0]) > nfb::smp::kMaxRuns) return NFB_ERR_UNSUPPORTED;
  NFB_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long N = (long long)map->height * map->width;
  if (!h->smp_runs) NFB_CUDA(dev_alloc(&h->smp_runs, nfb::smp::kMaxRuns));
  if (!h->smp_segs) NFB_CUDA(dev_alloc(&h->smp_segs, nfb::smp::kMaxSegs));
  if (h->smp_first_n < N) {
    if (h->smp_first) NFB_CUDA(cudaFree(h->smp_first));
    h->smp_first = nullptr; h->smp_first_n = 0;
    NFB_CUDA(dev_alloc(&h->smp_first, (size_t)N));
    h->smp_first_n = N;
    NFB_CUDA(nfb::launch_fill_int(h->smp_first, N, 0x7FFFFFFF, st, &h->launches));
  }
  nfb::SampleArgs a;
  std::memset(&a, 0, sizeof(a));
  a.map.H = map->height; a.map.W = map->width;
  a.map.b0 = map->bbox[0]; a.map.b1 = map->bbox[1]; a.map.b2 = map->bbox[2]; a.map.b3 = map->bbox[3];
  a.map.q_out = map->q_out; a.map.q_in = map->q_in;
  a.draws = draws; a.size = size; a.max_rounds = max_rounds; a.found = indices; a.state = state;
  a.runs = h->smp_runs; a.segs = h->smp_segs; a.first_pos = h->smp_first;
  if (g) {
    if ((g->target && !g->image) || (g->background_out && !g->background) || (g->ray_origins && !g->ray_directions)) return NFB_ERR_INVALID;
    for (int i = 0; i < 12; ++i) a.pose[i] = g->pose[i];
    a.fx = static_cast<float>(g->intrinsics[0]);
    a.fy = static_cast<float>(g->intrinsics[1]);
    a.wcx = static_cast<float>(static_cast<double>(map->width) * g->intrinsics[2]);
    a.hcy = static_cast<float>(static_cast<double>(map->height) * g->intrinsics[3]);
    a.image = g->image; a.background = g->background; a.ray_o = g->ray_origins; a.ray_d = g->ray_directions;
    a.target = g->target; a.bg_out = g->background_out; a.pixel_rc = g->pixel_rc;
  }
  NFB_CUDA(nfb::launch_sample_rays(a, st, &h->launches));
  return NFB_OK;
}

int nfb_host_map_cdf(const NfbRayMap* map, const long long* zeroed_sorted, int n_zero, const long long* ks, int n, double* out) {
  if (!map || !ks || !out || n < 0 || n_zero < 0 || (n_zero && !zeroed_sorted)) return NFB_ERR_INVALID;
  nfb::smp::Map m;
  m.H = map->height; m.W = map->width; m.b0 = map->bbox[0]; m.b1 = map->bbox[1]; m.b2 = map->bbox[2]; m.b3 = map->bbox[3];
  m.q_out = map->q_out; m.q_in = map->q_in;
  if (nfb::smp::num_runs(m) > nfb::smp::kMaxRuns) return NFB_ERR_UNSUPPORTED;
  std::vector<nfb::smp::Run> runs(nfb::smp::kMaxRuns);
  std::vector<nfb::smp::Seg> segs(nfb::smp::kMaxSegs);
  int nr = 0, ns = 0;
  const double total = nfb::smp::build_tables(m, zeroed_sorted, n_zero, runs.data(), nr, segs.data(), ns);
  if (ns > nfb::smp::kMaxSegs) return NFB_ERR_UNSUPPORTED;
  const long long N = (long long)m.H * m.W;
  for (int i = 0; i < n; ++i) {
    if (ks[i] < -1 || ks[i] >= N) return NFB_ERR_INVALID;
    out[i] = ks[i] < 0 ? total : nfb::smp::cdf_at(ks[i], runs.data(), nr, segs.data(), zeroed_sorted, n_zero);
  }
  return NFB_OK;
}

int nfb_debug_schedule(int which, int index, uint32_t* out, int out_words) {
  if (index >= 0 && (!out || out_words < 10)) return -1;
  switch (which) {
    case 0: return nfb::debug_prog_v4(index, out);
    case 1: return nfb::debug_prog_v6(index, out);
    case 2: return nfb::debug_prog_chain(index, out);
    case 3: return nfb::debug_jobs_dw(index, out);
    case 4: return index < 0 ? 1 : nfb::debug_dw_split(out);  // in/out: {num_sms, tiles 0, tiles 1} -> {parts0, parts1, groups}
    case 5: return nfb::debug_prog_chain_exact(index, out);
    case 6: return nfb::debug_stages_dw_exact(index, out);
    default:
      if (which >= 1000) {  // 1000 + n_iter * 100 + Tc * 10 + Tf: the pipelined kernel's job sequence
        const int w = which - 1000;
        return nfb::debug_jobs_v7(w / 100, (w / 10) % 10, w % 10, index, out);
      }
      return -1;
  }
}

int nfb_launch_count(NfbHandle* h, long long* out) {
  if (!h || !out) return NFB_ERR_INVALID;
  *out = h->launches;
  return NFB_OK;
}

}  // extern "C"
