// nfb_render_common.cuh — code shared by the render kernels (nfb_render.cu: one tile in flight, both precision modes and
// the training variant; nfb_render2.cu: two tiles in flight; nfb_render3.cu: two tiles in flight, pipelined passes): the
// per-sample arithmetic that must match the reference bit for bit (ray constants, depths, positional encoding, colour /
// sigma, cdf, inverse-CDF sampling, sort), the epilogue arithmetic of one accumulator chunk, the per-ray compositing and the
// clustered launch.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math_constants.h>

#include "nfb_internal.h"
#include "nfb_ptx.cuh"

namespace nfb {

constexpr int kRayFloats = 40;  // o[3] d[3] dnorm valid bg[3] gidx PEd[24] dz pad[3]
struct RayP {  // per-ray constants in shared memory (kRayFloats floats)
  float o[3], d[3];
  float dnorm;
  int valid;
  float bg[3];
  int gidx;
  float ped[24];
  float dz;
  float pad[3];
};
static_assert(sizeof(RayP) == kRayFloats * 4, "RayP size");

// Constants of ray g: origin and direction (explicit, or get_ray_bundle in-kernel), |d|, background and the direction
// encoder's d_z.  Rays beyond n_rays are marked invalid and zeroed.
__device__ __forceinline__ void load_ray(const RenderParams& p, int g, RayP& rp) {
  rp.valid = g < p.n_rays;
  rp.gidx = g;
  if (rp.valid) {
    float o0, o1, o2, d0, d1, d2;
    if (p.o) {
      o0 = p.o[3 * g]; o1 = p.o[3 * g + 1]; o2 = p.o[3 * g + 2];
      d0 = p.d[3 * g]; d1 = p.d[3 * g + 1]; d2 = p.d[3 * g + 2];
    } else {  // get_ray_bundle (nerf_helpers.py:111-122), same operation order in FP32
      const int pj = p.row_begin + g / p.width, pi = g % p.width;
      const float cx = __fdiv_rn(__fsub_rn((float)pi, p.wcx), p.fx);
      const float cy = -__fdiv_rn(__fsub_rn((float)pj, p.hcy), p.fy);
      d0 = __fadd_rn(__fadd_rn(__fmul_rn(cx, p.pose[0]), __fmul_rn(cy, p.pose[1])), __fmul_rn(-1.f, p.pose[2]));
      d1 = __fadd_rn(__fadd_rn(__fmul_rn(cx, p.pose[4]), __fmul_rn(cy, p.pose[5])), __fmul_rn(-1.f, p.pose[6]));
      d2 = __fadd_rn(__fadd_rn(__fmul_rn(cx, p.pose[8]), __fmul_rn(cy, p.pose[9])), __fmul_rn(-1.f, p.pose[10]));
      o0 = p.pose[3]; o1 = p.pose[7]; o2 = p.pose[11];
    }
    rp.o[0] = o0; rp.o[1] = o1; rp.o[2] = o2;
    rp.d[0] = d0; rp.d[1] = d1; rp.d[2] = d2;
    rp.dnorm = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(d0, d0), __fmul_rn(d1, d1)), __fmul_rn(d2, d2)));
    if (p.bg) { rp.bg[0] = p.bg[3 * g]; rp.bg[1] = p.bg[3 * g + 1]; rp.bg[2] = p.bg[3 * g + 2]; }
    rp.dz = p.dir_z ? p.dir_z[g] : d2;
  } else {
    for (int k = 0; k < 3; ++k) { rp.o[k] = 0.f; rp.d[k] = 0.f; rp.bg[k] = 0.f; }
    rp.dnorm = 0.f;
    rp.dz = 0.f;
  }
}

// Direction encoder input of ray slots [0, n): (d_z, near, far), as run_network reads ray_batch[..., -3:]
// (train_utils.py:14).  Thread tid < 12 n computes one accurate sincos.
__device__ __forceinline__ void dir_encoding(const RenderParams& p, RayP* rayp, int n, int tid) {
  if (tid < n * 12) {
    const int rr = tid / 12, k = tid - rr * 12, f = k / 3, c = k - f * 3;
    RayP& rp = rayp[rr];
    const float v = (c == 0) ? rp.dz : (c == 1 ? p.near_ : p.far_);
    float sn, cs;
    sincosf(v * (float)(1 << f), &sn, &cs);
    rp.ped[6 * f + c] = rp.valid ? sn : 0.f;
    rp.ped[6 * f + 3 + c] = rp.valid ? cs : 0.f;
  }
}

// Depth of coarse sample i (of nc == p.nc, which callers hold in a register) of ray rp (train_utils.py:56-76): linspace(near,
// far), with perturb jittered inside the sample's bin of mid-points.
__device__ __forceinline__ float coarse_depth(const RenderParams& p, const RayP& rp, int i, int nc) {
  const float tc = p.t_coarse[i];
  float z = __fadd_rn(__fmul_rn(p.near_, __fsub_rn(1.f, tc)), __fmul_rn(p.far_, tc));
  if (p.perturb) {
    float lower = z, upper = z;
    if (i > 0) {
      const float tp = p.t_coarse[i - 1];
      const float zp = __fadd_rn(__fmul_rn(p.near_, __fsub_rn(1.f, tp)), __fmul_rn(p.far_, tp));
      lower = __fmul_rn(0.5f, __fadd_rn(z, zp));
    }
    if (i < nc - 1) {
      const float tn = p.t_coarse[i + 1];
      const float zn = __fadd_rn(__fmul_rn(p.near_, __fsub_rn(1.f, tn)), __fmul_rn(p.far_, tn));
      upper = __fmul_rn(0.5f, __fadd_rn(zn, z));
    }
    const float tr = rp.valid ? p.t_rand[(size_t)rp.gidx * p.nc + i] : 0.f;
    z = __fadd_rn(lower, __fmul_rn(__fsub_rn(upper, lower), tr));
  }
  return z;
}

// ------------------------------------------------------------------------------------------------
// sin/cos of y for the positional encoding.  The reference evaluates torch.sin(x * 2^k) in FP32
// (nerf_helpers.py:231-233); x * 2^k is exact, so both variants see the same argument.
//   exact: libdevice sinf/cosf (<= 2 ulp).
//   fast : two-constant Cody-Waite reduction to [-pi, pi] + MUFU.SIN/COS (abs err ~5e-7), well below the
//          FP16 rounding (2.4e-4) the value then receives.
template <bool EXACT>
__device__ __forceinline__ void pe_sincos(float y, float& s, float& c) {
  if constexpr (EXACT) {
    sincosf(y, &s, &c);
  } else {
    const float n = rintf(y * 0.15915494309189535f);
    float r = fmaf(-n, 6.2831854820251465f, y);
    r = fmaf(-n, -1.7484555e-7f, r);
    s = __sinf(r);
    c = __cosf(r);
  }
}

// Positional encoding of the sample at depth z on ray rp (nerf_helpers.py:195-239): 63 lanes + 1 zero pad, of which the
// thread with lane half ch computes lanes [32 ch, 32 ch + 32).
template <bool EXACT>
__device__ __forceinline__ void pe_lanes(const RayP& rp, float z, int ch, float (&f)[32]) {
  const float px = __fadd_rn(rp.o[0], __fmul_rn(rp.d[0], z));
  const float py = __fadd_rn(rp.o[1], __fmul_rn(rp.d[1], z));
  const float pz = __fadd_rn(rp.o[2], __fmul_rn(rp.d[2], z));
  if (ch == 0) {  // lanes 0..31: xyz, frequencies 0..3, sin of frequency 4, cos(x), cos(y) of frequency 4
    f[0] = px; f[1] = py; f[2] = pz;
#pragma unroll
    for (int fr = 0; fr < 4; ++fr) {
      const float sc = (float)(1 << fr);
      pe_sincos<EXACT>(px * sc, f[3 + 6 * fr + 0], f[3 + 6 * fr + 3]);
      pe_sincos<EXACT>(py * sc, f[3 + 6 * fr + 1], f[3 + 6 * fr + 4]);
      pe_sincos<EXACT>(pz * sc, f[3 + 6 * fr + 2], f[3 + 6 * fr + 5]);
    }
    float cz;
    pe_sincos<EXACT>(px * 16.f, f[27], f[30]);
    pe_sincos<EXACT>(py * 16.f, f[28], f[31]);
    pe_sincos<EXACT>(pz * 16.f, f[29], cz);
  } else {        // lanes 32..63: cos(z) of frequency 4, frequencies 5..9, zero pad
    float sz;
    pe_sincos<EXACT>(pz * 16.f, sz, f[0]);
#pragma unroll
    for (int fr = 5; fr < 10; ++fr) {
      const float sc = (float)(1 << fr);
      const int b = 6 * fr - 29;  // lane 3 + 6*fr, minus 32
      pe_sincos<EXACT>(px * sc, f[b + 0], f[b + 3]);
      pe_sincos<EXACT>(py * sc, f[b + 1], f[b + 4]);
      pe_sincos<EXACT>(pz * sc, f[b + 2], f[b + 5]);
    }
    f[31] = 0.f;
  }
}

// FP16 of this thread's 32 encoding lanes (EXACT: hi in pe_hi, the remainder in pe_lo) -> row `row` of the 128-byte-swizzled
// PE buffer(s).
template <bool EXACT>
__device__ __forceinline__ void store_pe_row(const float (&f)[32], uint8_t* pe_hi, uint8_t* pe_lo, int row, int ch) {
#pragma unroll
  for (int qq = 0; qq < 4; ++qq) {
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float a = f[qq * 8 + 2 * e], b = f[qq * 8 + 2 * e + 1];
      hi[e] = pack_f16x2(a, b);
      if constexpr (EXACT) {
        const float2 hf = unpack_f16x2(hi[e]);
        lo[e] = pack_f16x2(a - hf.x, b - hf.y);
      }
    }
    const int off = row * 128 + (((ch * 4 + qq) ^ (row & 7)) << 4);
    *reinterpret_cast<uint4*>(pe_hi + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    if constexpr (EXACT) *reinterpret_cast<uint4*>(pe_lo + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

// (a0, a1) += (b0, b1) as one packed FP32 add (sm_100 FADD2; round-to-nearest per element, like two scalar adds).
__device__ __forceinline__ void add_f32x2(float& a0, float& a1, float b0, float b1) {
  asm("{\n\t.reg .b64 ra, rb, rc;\n\tmov.b64 ra, {%0, %1};\n\tmov.b64 rb, {%2, %3};\n\tadd.rn.f32x2 rc, ra, rb;\n\t"
      "mov.b64 {%0, %1}, rc;\n\t}"
      : "+f"(a0), "+f"(a1)
      : "f"(b0), "f"(b1));
}

// ------------------------------------------------------------------------------------------------
// Epilogue math of one 32-column accumulator chunk: x = acc + bias (+ extra); ReLU; FP16 hi (and lo).
template <bool EXACT>
__device__ __forceinline__ void epi_math(const uint32_t (&v)[32], uint32_t bias, uint32_t extra,
                                         float* __restrict__ dump, uint32_t (&hi)[16], uint32_t (&lo)[16]) {
  float x[32];  // bias / extra are shared-memory byte addresses (extra == 0: none)
#pragma unroll
  for (int j = 0; j < 32; j += 4) {  // packed FP32 adds (FADD2): same rounding as scalar adds, half the issue slots
    const float4 b = lds128(bias + j * 4);
    x[j] = __uint_as_float(v[j]); x[j + 1] = __uint_as_float(v[j + 1]);
    x[j + 2] = __uint_as_float(v[j + 2]); x[j + 3] = __uint_as_float(v[j + 3]);
    add_f32x2(x[j], x[j + 1], b.x, b.y);
    add_f32x2(x[j + 2], x[j + 3], b.z, b.w);
  }
  if (extra) {
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      const float4 e = lds128(extra + j * 4);
      add_f32x2(x[j], x[j + 1], e.x, e.y);
      add_f32x2(x[j + 2], x[j + 3], e.z, e.w);
    }
  }
  if (dump) {
#pragma unroll
    for (int j = 0; j < 32; ++j) dump[j] = fmaxf(x[j], 0.f);
  }
#pragma unroll
  for (int j = 0; j < 32; j += 2) {
    if constexpr (EXACT) {
      const float a = fmaxf(x[j], 0.f), b = fmaxf(x[j + 1], 0.f);
      hi[j / 2] = pack_f16x2(a, b);
      const float2 h = unpack_f16x2(hi[j / 2]);
      lo[j / 2] = pack_f16x2(a - h.x, b - h.y);
    } else {
      hi[j / 2] = pack_relu_f16x2(x[j], x[j + 1]);  // ReLU fused into the conversion
    }
  }
}

// ReLU mask of 32 post-activation FP16 values (bit j = feature j is non-zero).  An activation that is positive in FP32
// but rounds to FP16 zero counts as inactive: its value is what the next layer saw.
__device__ __forceinline__ uint32_t relu_mask32(const uint32_t (&h)[16]) {
  uint32_t m = 0u;
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    m |= ((h[j] & 0xFFFFu) ? 1u : 0u) << (2 * j);
    m |= ((h[j] >> 16) ? 1u : 0u) << (2 * j + 1);
  }
  return m;
}

__device__ __forceinline__ uint32_t cta_rank_early() { return cluster_ctarank(); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------------------------------------
// Compositing of one ray by one warp (volume_rendering_utils.py:7-75).  Samples are lane-blocked.  `pre`
// holds what the step-9 epilogue prepared per sample: (colour r, g, b, sigma) with colour = sigmoid(rgb raw)
// — or the raw background colour on the last sample (:29-33) — and sigma = relu(raw + noise) (+1e-6 on the
// last sample, :52-53).  Returns w of the last sample; lane 0 writes rgb[3], disp, acc.
__device__ __forceinline__ float composite_ray(const float4* __restrict__ pre, const float* __restrict__ z, float* __restrict__ wbuf,
                                               int S, float dnorm, bool white_bkgd, float* out_rgb, float* out_disp,
                                               float* out_acc, int lane) {
  const int per = (S + 31) >> 5;
  const int i0 = lane * per;
  // pass 1: alpha per sample (kept in wbuf), product of (1 - alpha + 1e-10) over this lane's block
  float prod = 1.f;
  for (int j = 0; j < per; ++j) {
    const int i = i0 + j;
    if (i < S) {
      float delta = (i < S - 1) ? __fsub_rn(z[i + 1], z[i]) : 1e10f;
      delta = __fmul_rn(delta, dnorm);
      const float alpha = __fsub_rn(1.f, expf(-__fmul_rn(pre[i].w, delta)));
      wbuf[i] = alpha;
      prod *= __fadd_rn(__fsub_rn(1.f, alpha), 1e-10f);
    }
  }
  // exclusive multiplicative scan over lanes
  float incl = prod;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl *= t;
  }
  float T = __shfl_up_sync(0xffffffffu, incl, 1);
  if (lane == 0) T = 1.f;
  // pass 2: weights and weighted sums
  float r = 0.f, g = 0.f, b = 0.f, depth = 0.f, acc = 0.f, wl = 0.f;
  for (int j = 0; j < per; ++j) {
    const int i = i0 + j;
    if (i < S) {
      const float alpha = wbuf[i];
      const float w = __fmul_rn(alpha, T);
      T *= __fadd_rn(__fsub_rn(1.f, alpha), 1e-10f);
      wbuf[i] = w;
      const float4 q = pre[i];
      r = fmaf(w, q.x, r); g = fmaf(w, q.y, g); b = fmaf(w, q.z, b);
      depth = fmaf(w, z[i], depth);
      acc += w;
      if (i == S - 1) wl = w;
    }
  }
  r = warp_sum(r); g = warp_sum(g); b = warp_sum(b);
  depth = warp_sum(depth); acc = warp_sum(acc); wl = warp_sum(wl);
  if (lane == 0 && out_rgb) {
    if (white_bkgd) { r += 1.f - acc; g += 1.f - acc; b += 1.f - acc; }
    out_rgb[0] = r; out_rgb[1] = g; out_rgb[2] = b;
    *out_disp = 1.f / fmaxf(1e-10f, depth / acc);
    *out_acc = acc;
  }
  return wl;
}

// fc_rgb output of sample i (of S) of ray rp in `pass` -> what compositing needs (volume_rendering_utils.py:29-33, 41-53):
// colour = sigmoid(raw rgb), or the background on the last sample; sigma = relu(raw sigma + noise), +1e-6 on the last
// sample.  has_bg: p.bg is set (a loop-invariant the callers keep in a register).  sig_in receives what the ReLU sees.
__device__ __forceinline__ float4 colour_sigma(const RenderParams& p, const RayP& rp, bool has_bg, float r0, float r1, float r2,
                                               float sigma_raw, int pass, int S, int i, float& sig_in) {
  float sig = sigma_raw;
  if (p.noise_std > 0.f && rp.valid)
    sig = __fadd_rn(sig, __fmul_rn((pass ? p.noise_f : p.noise_c)[(size_t)rp.gidx * S + i], p.noise_std));
  sig_in = sig;  // volume_rendering_utils.py:52
  sig = fmaxf(sig, 0.f);
  float4 pre;
  if (i == S - 1) {
    sig = __fadd_rn(sig, 1e-6f);
    if (has_bg) { pre.x = rp.bg[0]; pre.y = rp.bg[1]; pre.z = rp.bg[2]; }
  }
  if (!(has_bg && i == S - 1)) {
    pre.x = 1.f / (1.f + expf(-r0));
    pre.y = 1.f / (1.f + expf(-r1));
    pre.z = 1.f / (1.f + expf(-r2));
  }
  pre.w = sig;
  return pre;
}

// Inverse-CDF resampling, first half (sample_pdf_2, nerf_helpers.py:344-362), for one ray by one warp: the mid-point bins
// of the nc coarse depths z and the cdf over weights[1:-1] + 1e-5 (nc - 1 entries each).
__device__ __forceinline__ void build_cdf(const float* w, const float* z, float* cdf, float* bins, int nc, int lane) {
  const int nb = nc - 1;  // bins / cdf entries
  const int nw = nc - 2;  // interior weights
  for (int k = lane; k < nb; k += 32) bins[k] = __fmul_rn(0.5f, __fadd_rn(z[k + 1], z[k]));
  const int per = (nw + 31) >> 5;
  const int k0 = lane * per;
  float part = 0.f;
  for (int j = 0; j < per; ++j)
    if (k0 + j < nw) part += __fadd_rn(w[k0 + j + 1], 1e-5f);
  const float total = warp_sum(part);
  float psum = 0.f;
  for (int j = 0; j < per; ++j)
    if (k0 + j < nw) psum += __fdiv_rn(__fadd_rn(w[k0 + j + 1], 1e-5f), total);
  float incl = psum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float tt = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += tt;
  }
  float run = incl - psum;  // exclusive prefix of this lane's block
  if (lane == 0) cdf[0] = 0.f;
  for (int j = 0; j < per; ++j)
    if (k0 + j < nw) {
      run += __fdiv_rn(__fadd_rn(w[k0 + j + 1], 1e-5f), total);
      cdf[k0 + j + 1] = run;
    }
}

// Inverse-CDF resampling, second half (nerf_helpers.py:363-387): the depth of the sample drawn at u from nb cdf entries / bins.
__device__ __forceinline__ float sample_pdf(const float* cdf, const float* bins, int nb, float u) {
  int lo = 0, hi = nb;  // searchsorted(..., right=True): number of cdf entries <= u
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (cdf[mid] <= u) lo = mid + 1; else hi = mid;
  }
  const int below = max(0, lo - 1), above = min(nb - 1, lo);
  const float cb = cdf[below], ca = cdf[above];
  float den = __fsub_rn(ca, cb);
  if (den < 1e-5f) den = 1.f;
  const float tt = __fdiv_rn(__fsub_rn(u, cb), den);
  return __fadd_rn(bins[below], __fmul_rn(tt, __fsub_rn(bins[above], bins[below])));
}

// torch.sort(cat(z, z_samples)) (train_utils.py:126) as a rank merge: the position of element i of z = cat(nc coarse depths,
// nf samples) in the sorted array.  The coarse depths are sorted, the samples need not be (stochastic u), so an element's
// rank = (# coarse before it, by binary search) + (# samples before it, counted).  Ties: coarse first, then samples by
// index — equal values make any tie order give the same sorted array.
__device__ __forceinline__ int merge_rank(const float* z, int nc, int nf, int i) {
  const float* zs = z + nc;
  const float v = z[i];
  int rank;
  if (i < nc) {
    rank = i;
    for (int j = 0; j < nf; ++j) rank += (zs[j] < v) ? 1 : 0;
  } else {
    const int jm = i - nc;
    int lo = 0, hi = nc;  // # coarse depths <= v
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (z[mid] <= v) lo = mid + 1; else hi = mid;
    }
    rank = lo;
    for (int j = 0; j < nf; ++j) {
      const float y = zs[j];
      rank += (y < v || (y == v && j < jm)) ? 1 : 0;
    }
  }
  return rank;
}

// One launch of a render kernel on whole clusters of `cluster` CTAs: a CTA per unit of work (p.n_units), at most num_sms.
template <class Kernel>
cudaError_t launch_clustered(Kernel kernel, const RenderParams& p, int cluster, int threads, int smem_bytes, int num_sms,
                             cudaStream_t st, long long* launches) {
  int grid = p.n_units < num_sms ? p.n_units : num_sms;
  if (grid <= 0) return cudaSuccess;
  grid = (grid + cluster - 1) / cluster * cluster;
  if (grid > num_sms) grid = num_sms / cluster * cluster;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cluster;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, p);
  ++*launches;
  return e != cudaSuccess ? e : cudaGetLastError();
}


// Optional phase timers (NfbDebug.prof): cycles of one observer thread per role, summed over CTAs.  Compiled in only with
// -DNFB_TIMERS=1 (tools/phase_profile.py builds such a library): even disabled at run time they cost registers in the
// hot loops (measured: -15 % on the two-tile kernel).
#ifndef NFB_TIMERS
#define NFB_TIMERS 0
#endif
#if NFB_TIMERS
struct PhaseTimer {
  unsigned long long* dst;
  long long t0;
  __device__ __forceinline__ PhaseTimer(unsigned long long* d, bool on) : dst(on ? d : nullptr), t0(0) {
    if (dst) t0 = clock64();
  }
  __device__ __forceinline__ void lap(int slot) {
    if (dst) {
      const long long t1 = clock64();
      atomicAdd(dst + slot, (unsigned long long)(t1 - t0));
      t0 = t1;
    }
  }
};
#else
struct PhaseTimer {
  __device__ __forceinline__ PhaseTimer(unsigned long long*, bool) {}
  __device__ __forceinline__ void lap(int) {}
};
#endif

}  // namespace nfb
