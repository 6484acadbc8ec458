"""ctypes binding of include/nfb.h (lib/libnfb.so).  The library is REQUIRED: importing this module
raises if it is missing — there is no PyTorch or CPU fallback for the render path."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NFB_LIB") or os.path.join(os.path.dirname(_HERE), "lib", "libnfb.so")

NFB_OK = 0
NFB_NET_COARSE, NFB_NET_FINE = 0, 1
NFB_PREC_FAST, NFB_PREC_EXACT, NFB_PREC_EXACT_GRAD = 0, 1, 2

EXPORTS = ["nfb_version", "nfb_strerror", "nfb_last_cuda_error", "nfb_create", "nfb_destroy", "nfb_load_weights",
           "nfb_set_frame", "nfb_render_forward", "nfb_render_frame_host", "nfb_launch_count", "nfb_host_linspace",
           "nfb_render_forward_train", "nfb_render_backward", "nfb_train_debug", "nfb_debug_schedule", "nfb_loss_mse_grad",
           "nfb_adam_step", "nfb_adam_step_dev", "nfb_repack", "nfb_frame_products", "nfb_sample_rays", "nfb_host_map_cdf"]


class NfbModelDims(C.Structure):
    _fields_ = [("num_encoding_fn_xyz", C.c_int32), ("num_encoding_fn_dir", C.c_int32), ("include_input_xyz", C.c_int32),
                ("include_input_dir", C.c_int32), ("dim_expression", C.c_int32), ("dim_latent", C.c_int32)]


class NfbRays(C.Structure):
    _fields_ = [("o", C.c_void_p), ("d", C.c_void_p), ("n_rays", C.c_int32), ("pose", C.c_float * 12),
                ("intrinsics", C.c_double * 4), ("height", C.c_int32), ("width", C.c_int32), ("row_begin", C.c_int32),
                ("near_", C.c_float), ("far_", C.c_float), ("dir_z", C.c_void_p), ("background", C.c_void_p)]


class NfbSampling(C.Structure):
    _fields_ = [("num_coarse", C.c_int32), ("num_fine", C.c_int32), ("perturb", C.c_int32), ("noise_std", C.c_float),
                ("white_background", C.c_int32), ("lindisp", C.c_int32), ("precision", C.c_int32),
                ("t_coarse", C.c_void_p), ("u_fine", C.c_void_p)]


class NfbNoise(C.Structure):
    _fields_ = [("t_rand", C.c_void_p), ("sigma_noise_c", C.c_void_p), ("u", C.c_void_p), ("sigma_noise_f", C.c_void_p)]


class NfbOutputs(C.Structure):
    _fields_ = [("rgb_coarse", C.c_void_p), ("disp_coarse", C.c_void_p), ("acc_coarse", C.c_void_p),
                ("rgb_fine", C.c_void_p), ("disp_fine", C.c_void_p), ("acc_fine", C.c_void_p), ("w_last", C.c_void_p)]


class NfbDebug(C.Structure):
    _fields_ = [("z_coarse", C.c_void_p), ("raw_coarse", C.c_void_p), ("z_fine", C.c_void_p), ("raw_fine", C.c_void_p),
                ("act_dump", C.c_void_p), ("act_step", C.c_int32), ("prof", C.c_void_p)]


class NfbOutGrads(C.Structure):
    _fields_ = [("rgb_coarse", C.c_void_p), ("disp_coarse", C.c_void_p), ("acc_coarse", C.c_void_p),
                ("rgb_fine", C.c_void_p), ("disp_fine", C.c_void_p), ("acc_fine", C.c_void_p), ("w_last", C.c_void_p)]


class NfbTrainDebug(C.Structure):
    _fields_ = [("records", C.c_void_p), ("n_tiles", C.c_longlong), ("record_bytes", C.c_int32), ("d_raw", C.c_void_p),
                ("acc_coarse", C.c_void_p), ("acc_fine", C.c_void_p), ("acc_floats", C.c_int32), ("scale", C.c_void_p),
                ("z_coarse", C.c_void_p), ("raw_coarse", C.c_void_p), ("z_fine", C.c_void_p), ("raw_fine", C.c_void_p),
                ("tiles_coarse", C.c_int32), ("tiles_fine", C.c_int32), ("rays_per_unit", C.c_int32)]


class NfbAdam(C.Structure):
    _fields_ = [("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float), ("step", C.c_int32),
                ("grad_scale", C.c_float), ("reg_offset", C.c_longlong), ("reg_weight", C.c_float)]


class NfbAdamDev(C.Structure):
    _fields_ = [("step", C.c_int32), ("pad", C.c_int32), ("lr0", C.c_float), ("decay_factor", C.c_float), ("decay_steps", C.c_float),
                ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float), ("grad_scale", C.c_float), ("reg_weight", C.c_float),
                ("table_offset", C.c_longlong), ("row", C.c_void_p), ("lr_over_bc1", C.c_float), ("sqrt_bc2", C.c_float),
                ("reg_offset", C.c_longlong)]


class NfbRayMap(C.Structure):
    _fields_ = [("height", C.c_int32), ("width", C.c_int32), ("bbox", C.c_int32 * 4), ("q_out", C.c_double), ("q_in", C.c_double)]


class NfbRayGather(C.Structure):
    _fields_ = [("pose", C.c_float * 12), ("intrinsics", C.c_double * 4), ("image", C.c_void_p), ("background", C.c_void_p),
                ("ray_origins", C.c_void_p), ("ray_directions", C.c_void_p), ("target", C.c_void_p), ("background_out", C.c_void_p),
                ("pixel_rc", C.c_void_p)]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} not found: build it with `python 4d-facial-avatars_b200/build.py` "
                          "(the render path has no fallback)")
    lib = C.CDLL(LIB_PATH)
    lib.nfb_version.restype = C.c_int
    lib.nfb_strerror.restype = C.c_char_p
    lib.nfb_strerror.argtypes = [C.c_int]
    lib.nfb_last_cuda_error.restype = C.c_char_p
    lib.nfb_create.argtypes = [C.POINTER(NfbModelDims), C.c_int, C.POINTER(C.c_void_p)]
    lib.nfb_destroy.argtypes = [C.c_void_p]
    lib.nfb_load_weights.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_void_p]
    lib.nfb_set_frame.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.nfb_render_forward.argtypes = [C.c_void_p, C.POINTER(NfbRays), C.POINTER(NfbSampling), C.POINTER(NfbNoise),
                                       C.POINTER(NfbOutputs), C.POINTER(NfbDebug), C.c_void_p]
    lib.nfb_render_frame_host.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_double), C.c_int, C.c_int, C.c_int,
                                          C.c_int, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.POINTER(NfbSampling), C.c_void_p, C.c_void_p]
    lib.nfb_render_forward_train.argtypes = [C.c_void_p, C.POINTER(NfbRays), C.POINTER(NfbSampling), C.POINTER(NfbNoise),
                                             C.POINTER(NfbOutputs), C.c_void_p]
    lib.nfb_render_backward.argtypes = [C.c_void_p, C.POINTER(NfbOutGrads), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                        C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p]
    lib.nfb_train_debug.argtypes = [C.c_void_p, C.POINTER(NfbTrainDebug)]
    lib.nfb_loss_mse_grad.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_longlong, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p]
    lib.nfb_adam_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.POINTER(NfbAdam), C.c_void_p]
    lib.nfb_adam_step_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p]
    lib.nfb_repack.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_void_p]
    lib.nfb_frame_products.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_double), C.c_int, C.c_int,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    lib.nfb_sample_rays.argtypes = [C.c_void_p, C.POINTER(NfbRayMap), C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                    C.POINTER(NfbRayGather), C.c_void_p]
    lib.nfb_host_map_cdf.argtypes = [C.POINTER(NfbRayMap), C.POINTER(C.c_longlong), C.c_int, C.POINTER(C.c_longlong), C.c_int,
                                     C.POINTER(C.c_double)]
    lib.nfb_launch_count.argtypes = [C.c_void_p, C.POINTER(C.c_longlong)]
    lib.nfb_host_linspace.argtypes = [C.POINTER(C.c_float), C.c_int]
    for fn in ("nfb_create", "nfb_destroy", "nfb_load_weights", "nfb_set_frame", "nfb_render_forward",
               "nfb_render_frame_host", "nfb_launch_count", "nfb_host_linspace", "nfb_render_forward_train",
               "nfb_render_backward", "nfb_train_debug", "nfb_loss_mse_grad", "nfb_adam_step", "nfb_adam_step_dev", "nfb_repack", "nfb_frame_products",
               "nfb_sample_rays", "nfb_host_map_cdf"):
        getattr(lib, fn).restype = C.c_int
    return lib


lib = _load()


def check(rc, what=""):
    if rc != NFB_OK:
        msg = lib.nfb_strerror(rc).decode()
        detail = lib.nfb_last_cuda_error().decode()
        raise RuntimeError(f"nfb {what}: {msg}" + (f" [{detail}]" if detail and rc == 3 else ""))
