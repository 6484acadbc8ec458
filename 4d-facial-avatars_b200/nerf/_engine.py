"""Host-side engine: owns NfbHandle objects, keeps the packed weight streams in sync with the caller's
FP32 nn.Parameters, and launches the fused render kernel on torch's current CUDA stream.

torch is used here only for device memory, streams and (in the trainer) torch.distributed."""
import ctypes as C
import os
import weakref

import torch

from . import _capi as capi

PARAM_ORDER = ([f"layers_xyz.{i}.{k}" for i in range(6) for k in ("weight", "bias")]
               + ["fc_feat.weight", "fc_feat.bias", "fc_alpha.weight", "fc_alpha.bias"]
               + [f"layers_dir.{i}.{k}" for i in range(4) for k in ("weight", "bias")]
               + ["fc_rgb.weight", "fc_rgb.bias"])

_precision = os.environ.get("NFB_PRECISION", "fast")
_PREC_CODES = {"fast": capi.NFB_PREC_FAST, "exact": capi.NFB_PREC_EXACT, "exact_grad": capi.NFB_PREC_EXACT_GRAD}


def set_precision(mode: str):
    """'fast' = FP16 operands / FP32 accumulate; 'exact' = 3-pass FP16 hi/lo split of the forward (see include/nfb.h);
    'exact_grad' = 'exact', and training gradients computed from hi/lo operands as well (twice the record memory)."""
    global _precision
    if mode not in _PREC_CODES:
        raise ValueError("precision must be 'fast', 'exact' or 'exact_grad'")
    _precision = mode


def _prec_code(prec):
    return _PREC_CODES.get(prec, capi.NFB_PREC_FAST)


def get_precision() -> str:
    return _precision


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32c(t, device):
    return t.detach().to(device=device, dtype=torch.float32).contiguous()


class Renderer:
    """One NfbHandle on one CUDA device plus the bookkeeping that decides when weights must be re-packed."""

    def __init__(self, device: torch.device):
        if device.type != "cuda":
            raise RuntimeError("the nfb render path runs on CUDA (sm_100a) only; there is no CPU fallback")
        self.device = device
        idx = device.index if device.index is not None else torch.cuda.current_device()
        dims = capi.NfbModelDims(10, 4, 1, 0, 76, 32)
        h = C.c_void_p()
        capi.check(capi.lib.nfb_create(C.byref(dims), idx, C.byref(h)), "create")
        self._h = h
        self._lin = {}
        self._plist = {}
        self.packed_owner = None   # the FusedTrainer whose weights the packed streams hold (None: whatever sync_weights packed last)
        self._versions = [None, None]
        self._keep = [None, None]  # contiguous FP32 copies handed to the pack kernels
        self.train_token = 0       # bumped by every training forward: the handle keeps ONE saved state
        weakref.finalize(self, capi.lib.nfb_destroy, h)

    def _params(self, model):
        """The model's 26 parameters in PARAM_ORDER; the walk over named_parameters() is cached per module object."""
        cached = self._plist.get(id(model))
        if cached is None or cached[0]() is not model:
            sd = dict(model.named_parameters())
            cached = self._plist[id(model)] = (weakref.ref(model), [sd[k] for k in PARAM_ORDER])
        return cached[1]

    def _fingerprint(self, model):
        """(identity, storage, in-place version) of every parameter.  Writes that bypass autograd's version counter
        (`p.data.copy_()`, external kernels) are invisible here: call invalidate() after them."""
        return (id(model),) + tuple((p.data_ptr(), p._version) for p in self._params(model))

    def invalidate(self):
        """Force a re-pack of both networks at the next render (after parameter writes torch cannot see)."""
        self._versions = [None, None]

    def mark_synced(self, model_coarse, model_fine):
        """The packed streams already hold these models' current values (the fused optimizer step re-packed them)."""
        self._versions[0] = self._fingerprint(model_coarse)
        if model_fine is not None:
            self._versions[1] = self._fingerprint(model_fine)

    def sync_weights(self, model_coarse, model_fine):
        for which, model in ((capi.NFB_NET_COARSE, model_coarse), (capi.NFB_NET_FINE, model_fine)):
            if model is None:
                continue
            fp = self._fingerprint(model)
            if fp == self._versions[which]:
                continue
            tensors = [_f32c(t, self.device) for t in self._params(model)]
            arr = (C.c_void_p * 26)(*[t.data_ptr() for t in tensors])
            capi.check(capi.lib.nfb_load_weights(self._h, which, arr, _stream()), "load_weights")
            self.packed_owner = None
            self._keep[which] = tensors
            self._versions[which] = fp

    def linspace(self, n):
        """torch.linspace(0, 1, n) evaluated by ATen's CPU kernel (whose vectorised halves are not the scalar
        formula of nfb_host_linspace) and cached on the device, so depths match the CPU reference bit for bit."""
        t = self._lin.get(n)
        if t is None:
            t = self._lin[n] = torch.linspace(0.0, 1.0, n, dtype=torch.float32).to(self.device)
        return t

    def set_frame(self, expressions, latent_code):
        e = _f32c(expressions, self.device).reshape(-1)
        l = _f32c(latent_code, self.device).reshape(-1)
        if e.numel() != 76 or l.numel() != 32:
            raise ValueError("expressions must have 76 and latent_code 32 elements")
        capi.check(capi.lib.nfb_set_frame(self._h, _ptr(e), _ptr(l), _stream()), "set_frame")
        self._frame = (e, l)

    def kernel_info(self, precision="fast"):
        """Which render kernel an evaluation call in this precision runs, and the ncu capture that describes it (bench.py)."""
        k = os.environ.get("NFB_KERNEL", "")
        if precision != "fast" or k == "v4":
            return dict(name="nfb::render_kernel", block_size=320, ncu_json="r2_render_kernel_exact_ncu.json")
        if k == "v6":
            return dict(name="nfb::v6::render2_kernel", block_size=384, ncu_json="r2_render2_kernel_ncu.json")
        return dict(name="nfb::v7::render3_kernel", block_size=512, ncu_json="r2_render3_kernel_ncu.json")

    def launch_count(self) -> int:
        n = C.c_longlong()
        capi.check(capi.lib.nfb_launch_count(self._h, C.byref(n)))
        return n.value

    def render(self, ro, rd, near, far, num_coarse, num_fine, perturb=False, noise_std=0.0, white_bkgd=False,
               background=None, dir_z=None, noise=None, precision=None, debug=False, act_step=None, train=False):
        """ro, rd: [N,3] CUDA FP32.  noise: dict with t_rand, n_c, u, n_f (any may be None).  Returns a dict
        with the seven outputs (+ per-sample dumps when debug).  train=True: nfb_render_forward_train (the handle keeps
        the state `backward` consumes)."""
        dev = self.device
        ro, rd = _f32c(ro, dev), _f32c(rd, dev)
        n = ro.shape[0]
        has_fine = num_fine > 0
        out = {k: torch.empty((n, 3) if k.startswith("rgb") else (n,), device=dev, dtype=torch.float32)
               for k in ("rgb_coarse", "disp_coarse", "acc_coarse", "w_last")}
        if has_fine:
            out.update({k: torch.empty((n, 3) if k.startswith("rgb") else (n,), device=dev, dtype=torch.float32)
                        for k in ("rgb_fine", "disp_fine", "acc_fine")})
        rays = capi.NfbRays()
        rays.o, rays.d, rays.n_rays = ro.data_ptr(), rd.data_ptr(), n
        rays.near_, rays.far_ = float(near), float(far)
        keep = [ro, rd]
        if background is not None:
            bg = _f32c(background, dev).reshape(n, 3)
            rays.background = bg.data_ptr()
            keep.append(bg)
        if dir_z is not None:
            dz = _f32c(dir_z, dev).reshape(n)
            rays.dir_z = dz.data_ptr()
            keep.append(dz)
        prec = precision or _precision
        sm = capi.NfbSampling(num_coarse, num_fine, int(bool(perturb)), float(noise_std), int(bool(white_bkgd)), 0,
                              _prec_code(prec),
                              self.linspace(num_coarse).data_ptr(),
                              self.linspace(num_fine).data_ptr() if has_fine else None)
        nz = capi.NfbNoise()
        if noise:
            for field, key in (("t_rand", "t_rand"), ("sigma_noise_c", "n_c"), ("u", "u"), ("sigma_noise_f", "n_f")):
                t = noise.get(key)
                if t is not None:
                    t = _f32c(t, dev)
                    keep.append(t)
                    setattr(nz, field, t.data_ptr())
        o = capi.NfbOutputs(out["rgb_coarse"].data_ptr(), out["disp_coarse"].data_ptr(), out["acc_coarse"].data_ptr(),
                            out["rgb_fine"].data_ptr() if has_fine else None,
                            out["disp_fine"].data_ptr() if has_fine else None,
                            out["acc_fine"].data_ptr() if has_fine else None, out["w_last"].data_ptr())
        dbg = None
        if debug or act_step is not None:
            s = num_coarse + num_fine
            out["z_coarse"] = torch.zeros((n, num_coarse), device=dev)
            out["raw_coarse"] = torch.zeros((n, num_coarse, 4), device=dev)
            dbg = capi.NfbDebug(out["z_coarse"].data_ptr(), out["raw_coarse"].data_ptr(), None, None, None, 0)
            if has_fine:
                out["z_fine"] = torch.zeros((n, s), device=dev)
                out["raw_fine"] = torch.zeros((n, s, 4), device=dev)
                dbg.z_fine, dbg.raw_fine = out["z_fine"].data_ptr(), out["raw_fine"].data_ptr()
            if act_step is not None:
                out["act"] = torch.zeros((128, 256), device=dev)
                dbg.act_dump, dbg.act_step = out["act"].data_ptr(), int(act_step)
        if train:
            self.train_token += 1
            capi.check(capi.lib.nfb_render_forward_train(self._h, C.byref(rays), C.byref(sm), C.byref(nz) if noise else None,
                                                         C.byref(o), _stream()), "render_forward_train")
        else:
            capi.check(capi.lib.nfb_render_forward(self._h, C.byref(rays), C.byref(sm), C.byref(nz) if noise else None,
                                                   C.byref(o), C.byref(dbg) if dbg is not None else None, _stream()),
                       "render_forward")
        out["_keep"] = keep  # inputs must outlive the asynchronous launch
        return out

    def loss_mse_grad(self, rgb_c, rgb_f, target, n_total, grad_c, grad_f, loss):
        """nfb_loss_mse_grad: d mse / d rgb into grad_c / grad_f ([n,3] CUDA buffers), loss[0:2] += this shard's share."""
        n = rgb_c.shape[0]
        capi.check(capi.lib.nfb_loss_mse_grad(self._h, _ptr(rgb_c), _ptr(rgb_f), _ptr(target), n, int(n_total), _ptr(grad_c),
                                              _ptr(grad_f), _ptr(loss), _stream()), "loss_mse_grad")

    def adam_step(self, params, grads, exp_avg, exp_avg_sq, lr, step, betas=(0.9, 0.999), eps=1e-8, grad_scale=1.0,
                  reg_offset=-1, reg_weight=0.0):
        """nfb_adam_step over flat FP32 CUDA buffers (in place; grads are zeroed)."""
        hp = capi.NfbAdam(float(lr), float(betas[0]), float(betas[1]), float(eps), int(step), float(grad_scale), int(reg_offset),
                          float(reg_weight))
        capi.check(capi.lib.nfb_adam_step(self._h, _ptr(params), _ptr(grads), _ptr(exp_avg), _ptr(exp_avg_sq), params.numel(),
                                          C.byref(hp), _stream()), "adam_step")

    def adam_step_dev(self, params, grads, exp_avg, exp_avg_sq, dev_state):
        """nfb_adam_step_dev: like adam_step with step counter / LR schedule / regularised row in the device struct `dev_state`
        (a uint8 CUDA tensor holding an NfbAdamDev) — capturable in a CUDA graph."""
        capi.check(capi.lib.nfb_adam_step_dev(self._h, _ptr(params), _ptr(grads), _ptr(exp_avg), _ptr(exp_avg_sq), params.numel(),
                                              _ptr(dev_state), _stream()), "adam_step_dev")

    def repack(self, params_c, params_f):
        """nfb_repack: both networks' FP32 parameter tensors (lists in PARAM_ORDER) -> kernel-layout streams, one launch."""
        pc = (C.c_void_p * 26)(*[t.data_ptr() for t in params_c])
        pf = (C.c_void_p * 26)(*[t.data_ptr() for t in params_f]) if params_f is not None else None
        capi.check(capi.lib.nfb_repack(self._h, pc, pf, _stream()), "repack")

    def backward_into(self, out_grads, params_c, params_f, grads_c, grads_f, grad_latent):
        """nfb_render_backward writing straight into caller-owned gradient tensors (views of a flat bucket): params_* / grads_*
        are lists of 26 contiguous FP32 CUDA tensors in PARAM_ORDER (grads of layers_dir.3.* may be None)."""
        og = capi.NfbOutGrads()
        keep = []
        for field, g in zip(("rgb_coarse", "disp_coarse", "acc_coarse", "rgb_fine", "disp_fine", "acc_fine", "w_last"), out_grads):
            if g is not None:
                keep.append(g)
                setattr(og, field, g.data_ptr())
        arr = lambda ts: (C.c_void_p * 26)(*[(t.data_ptr() if t is not None else None) for t in ts]) if ts is not None else None  # noqa: E731
        capi.check(capi.lib.nfb_render_backward(self._h, C.byref(og), arr(params_c), arr(params_f), arr(grads_c), arr(grads_f),
                                                _ptr(grad_latent), _stream()), "render_backward")
        self._bwd_keep = keep

    def backward(self, out_grads, params_c, params_f, want_latent=True):
        """nfb_render_backward for the last training forward.  out_grads: 7 CUDA tensors or None (rgb_c, disp_c, acc_c,
        rgb_f, disp_f, acc_f, w_last); params_*: the 26 FP32 parameter tensors in PARAM_ORDER (params_f None without a
        fine network).  Returns (grads_c, grads_f, grad_latent) — lists aligned with PARAM_ORDER, None for layers_dir.3.*."""
        dev = self.device
        keep = []
        og = capi.NfbOutGrads()
        for field, g in zip(("rgb_coarse", "disp_coarse", "acc_coarse", "rgb_fine", "disp_fine", "acc_fine", "w_last"), out_grads):
            if g is not None:
                g = _f32c(g, dev)
                keep.append(g)
                setattr(og, field, g.data_ptr())

        def pack(params):
            if params is None:
                return None, None, None
            ps = [_f32c(t, dev) for t in params]
            gs = [None if PARAM_ORDER[i].startswith("layers_dir.3") else torch.empty_like(ps[i]) for i in range(26)]
            keep.extend(ps)
            return ((C.c_void_p * 26)(*[t.data_ptr() for t in ps]),
                    (C.c_void_p * 26)(*[(g.data_ptr() if g is not None else None) for g in gs]), gs)

        pc, gc, grads_c = pack(params_c)
        pf, gf, grads_f = pack(params_f)
        glat = torch.empty(32, device=dev, dtype=torch.float32) if want_latent else None
        capi.check(capi.lib.nfb_render_backward(self._h, C.byref(og), pc, pf, gc, gf, _ptr(glat), _stream()), "render_backward")
        self._bwd_keep = keep
        return grads_c, grads_f, glat

    def train_debug(self):
        d = capi.NfbTrainDebug()
        capi.check(capi.lib.nfb_train_debug(self._h, C.byref(d)), "train_debug")
        return d

    def render_camera(self, pose, intrinsics, height, width, row_begin, rows, near, far, num_coarse, num_fine,
                      background=None, out=None, precision=None, white_bkgd=False, prof=None):
        """Deterministic render of image rows [row_begin, row_begin+rows) with in-kernel ray generation
        (no o/d tensors in HBM).  pose: 3x4 / 4x4 CPU tensor; background: [rows*width,3] CUDA tensor or None.
        `out`: optional preallocated [11, rows*width] CUDA buffer; returns the dict of output views."""
        dev = self.device
        n = rows * width
        if out is None:
            out = torch.empty((11, n), device=dev, dtype=torch.float32)
        flat = out.view(-1)
        views = dict(rgb_coarse=flat[0:3 * n].view(n, 3), disp_coarse=flat[3 * n:4 * n], acc_coarse=flat[4 * n:5 * n],
                     rgb_fine=flat[5 * n:8 * n].view(n, 3), disp_fine=flat[8 * n:9 * n], acc_fine=flat[9 * n:10 * n],
                     w_last=flat[10 * n:11 * n])
        rays = capi.NfbRays()
        rays.n_rays = n
        p = pose.detach().cpu().float().reshape(-1)
        rows34 = p[:12] if p.numel() in (12, 16) else None
        for i in range(12):
            rays.pose[i] = float(rows34[i])
        for i in range(4):
            rays.intrinsics[i] = float(intrinsics[i])
        rays.height, rays.width, rays.row_begin = height, width, row_begin
        rays.near_, rays.far_ = float(near), float(far)
        if background is not None:
            rays.background = background.data_ptr()
        prec = precision or _precision
        has_fine = num_fine > 0
        sm = capi.NfbSampling(num_coarse, num_fine, 0, 0.0, int(bool(white_bkgd)), 0,
                              _prec_code(prec),
                              self.linspace(num_coarse).data_ptr(), self.linspace(num_fine).data_ptr() if has_fine else None)
        o = capi.NfbOutputs(views["rgb_coarse"].data_ptr(), views["disp_coarse"].data_ptr(), views["acc_coarse"].data_ptr(),
                            views["rgb_fine"].data_ptr() if has_fine else None,
                            views["disp_fine"].data_ptr() if has_fine else None,
                            views["acc_fine"].data_ptr() if has_fine else None, views["w_last"].data_ptr())
        dbg = None
        if prof is not None:  # int64[64] CUDA tensor of phase-cycle counters
            dbg = capi.NfbDebug()
            dbg.prof = prof.data_ptr()
        capi.check(capi.lib.nfb_render_forward(self._h, C.byref(rays), C.byref(sm), None, C.byref(o),
                                               C.byref(dbg) if dbg is not None else None, _stream()), "render_forward")
        views["_buf"] = out
        return views

    def render_frame_host(self, pose, intrinsics, height, width, row_begin, rows, near, far, expr_host, latent_host,
                          bg_host, num_coarse, num_fine, out_host, precision=None, white_bkgd=False):
        """Host-buffer end-to-end call (bench e2e leg).  All tensors are CPU (ideally pinned) FP32."""
        prec = precision or _precision
        sm = capi.NfbSampling(num_coarse, num_fine, 0, 0.0, int(bool(white_bkgd)), 0,
                              _prec_code(prec),
                              self.linspace(num_coarse).data_ptr(),
                              self.linspace(num_fine).data_ptr() if num_fine > 0 else None)
        pose_a = (C.c_float * 12)(*[float(v) for v in pose.reshape(-1)[:12]])
        intr_a = (C.c_double * 4)(*[float(v) for v in intrinsics])
        capi.check(capi.lib.nfb_render_frame_host(self._h, pose_a, intr_a, height, width, row_begin, rows, float(near),
                                                  float(far), _ptr(expr_host), _ptr(latent_host), _ptr(bg_host),
                                                  C.byref(sm), _ptr(out_host), _stream()), "render_frame_host")


_renderers = {}


def renderer_for(device: torch.device) -> Renderer:
    if device.type != "cuda":
        raise RuntimeError("the nfb render path runs on CUDA (sm_100a) only; there is no CPU fallback")
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    r = _renderers.get(key)
    if r is None:
        r = _renderers[key] = Renderer(torch.device("cuda", key[1]))
    return r
