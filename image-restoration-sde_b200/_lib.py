"""ctypes binding of libirsde_b200.so (the C ABI in include/irsde_b200.h).

There is no CPU or PyTorch fallback: if the library is missing, or there is no sm_100 device, calls
raise.  ``load()`` only dlopens (works without a GPU, used by the symbol-export test).
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("IRSDE_B200_LIB") or os.path.join(HERE, "libirsde_b200.so")  # override: A/B of builds

PREC_FP32, PREC_BF16, PREC_FP32X3 = 0, 1, 2
# name -> irsde_config.precision.  fp32: fp32 storage + SIMT FMA; bf16: tcgen05 bf16 (perf mode); fp32x3: fp32 storage,
# every conv = 3 x tcgen05.mma.kind::tf32 on hi/lo split operands (tensor cores at the fp32 mode's accuracy)
PRECISIONS = {"fp32": PREC_FP32, "bf16": PREC_BF16, "fp32x3": PREC_FP32X3}
NET_CONDITIONAL, NET_DENOISING = 0, 1
MODE_SDE, MODE_ODE, MODE_POSTERIOR, MODE_DSDE_SDE, MODE_DSDE_ODE = range(5)
NUM_COEF = 8
FLAG_FORCE_SIMT = 1   # irsde_config.flags: bf16 storage through the SIMT conv engine (debug aid)

# every symbol include/irsde_b200.h declares
SYMBOLS = ["irsde_create", "irsde_create_ch_mult", "irsde_create_nafnet", "irsde_create_nafnet_lens", "irsde_set_lens", "irsde_create_latent_unet", "irsde_latent_shape", "irsde_latent_encode",
           "irsde_latent_decode", "irsde_tensor2img_u8", "irsde_img2tensor_u8", "irsde_sqerr_u8", "irsde_ssim_workspace", "irsde_ssim_u8", "irsde_destroy", "irsde_last_error", "irsde_version", "irsde_load_tensor",
           "irsde_finalize_weights", "irsde_set_schedule", "irsde_set_coeffs", "irsde_noise_fn", "irsde_step",
           "irsde_reverse", "irsde_noise_state", "irsde_noise_state_images", "irsde_set_image_base", "irsde_set_image_uids", "irsde_comm_unique_id", "irsde_comm_init", "irsde_broadcast_weights", "irsde_gather", "irsde_launch_count", "irsde_device_bytes", "irsde_conv2d", "irsde_profile_begin",
           "irsde_profile_end", "irsde_profile_end_bytes", "irsde_conv2d_ex", "irsde_plan_num_ops", "irsde_plan_op_info", "irsde_trace_forward",
           "irsde_trim", "irsde_random_states"]


class Config(ctypes.Structure):
    _fields_ = [("in_nc", ctypes.c_int32), ("out_nc", ctypes.c_int32), ("nf", ctypes.c_int32),
                ("depth", ctypes.c_int32), ("variant", ctypes.c_int32), ("precision", ctypes.c_int32),
                ("device", ctypes.c_int32), ("flags", ctypes.c_int32)]


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "irsde_b200: %s not found. Build it with `python image-restoration-sde_b200/build.py` "
            "(needs nvcc with sm_100a support). There is no CPU / PyTorch fallback." % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    vp, i32, i64, u64, fp = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_uint64, ctypes.POINTER(ctypes.c_float)
    L.irsde_create.argtypes = [ctypes.POINTER(Config), ctypes.POINTER(vp)]
    L.irsde_create.restype = ctypes.c_int
    L.irsde_create_ch_mult.argtypes = [ctypes.POINTER(Config), ctypes.POINTER(i32), i32, ctypes.POINTER(vp)]
    L.irsde_create_ch_mult.restype = ctypes.c_int
    L.irsde_destroy.argtypes = [vp]
    L.irsde_destroy.restype = None
    L.irsde_last_error.argtypes = [vp]
    L.irsde_last_error.restype = ctypes.c_char_p
    L.irsde_version.argtypes = []
    L.irsde_version.restype = ctypes.c_char_p
    L.irsde_load_tensor.argtypes = [vp, ctypes.c_char_p, vp, i32, ctypes.POINTER(i64)]
    L.irsde_load_tensor.restype = ctypes.c_int
    L.irsde_finalize_weights.argtypes = [vp]
    L.irsde_finalize_weights.restype = ctypes.c_int
    L.irsde_set_schedule.argtypes = [vp, fp, fp, fp, fp, ctypes.c_float, ctypes.c_float, i32]
    L.irsde_set_schedule.restype = ctypes.c_int
    L.irsde_set_coeffs.argtypes = [vp, i32, fp, i32]
    L.irsde_set_coeffs.restype = ctypes.c_int
    L.irsde_noise_fn.argtypes = [vp, vp, vp, fp, i32, vp, i32, i32, i32, vp]
    L.irsde_noise_fn.restype = ctypes.c_int
    L.irsde_step.argtypes = [vp, i32, vp, vp, vp, vp, i32, vp, i64, vp]
    L.irsde_step.restype = ctypes.c_int
    L.irsde_reverse.argtypes = [vp, i32, vp, vp, vp, vp, i32, i32, i32, i32, u64, i32, vp]
    L.irsde_reverse.restype = ctypes.c_int
    L.irsde_noise_state.argtypes = [vp, vp, vp, i64, u64, vp]
    L.irsde_noise_state.restype = ctypes.c_int
    L.irsde_noise_state_images.argtypes = [vp, vp, vp, i32, i64, u64, vp]
    L.irsde_noise_state_images.restype = ctypes.c_int
    L.irsde_set_image_base.argtypes = [vp, u64]
    L.irsde_set_image_base.restype = ctypes.c_int
    L.irsde_set_image_uids.argtypes = [vp, ctypes.POINTER(ctypes.c_uint64), i32, vp]
    L.irsde_set_image_uids.restype = ctypes.c_int
    L.irsde_launch_count.argtypes = [vp]
    L.irsde_launch_count.restype = i64
    L.irsde_device_bytes.argtypes = [vp]
    L.irsde_device_bytes.restype = i64
    L.irsde_conv2d.argtypes = [vp, i32, vp, vp, vp, vp] + [i32] * 11 + [vp]
    L.irsde_conv2d.restype = ctypes.c_int
    L.irsde_conv2d_ex.argtypes = [vp, i32, vp, vp, vp, vp, vp] + [i32] * 12 + [vp]
    L.irsde_conv2d_ex.restype = ctypes.c_int
    L.irsde_plan_num_ops.argtypes = [vp, i32, i32, i32]
    L.irsde_plan_num_ops.restype = i32
    L.irsde_plan_op_info.argtypes = [vp, i32, i32, i32, i32, ctypes.c_char_p, i32, ctypes.POINTER(i32)]
    L.irsde_plan_op_info.restype = ctypes.c_int
    L.irsde_trace_forward.argtypes = [vp, vp, vp, fp, i32, i32, i32, i32, i32, vp, vp]
    L.irsde_trace_forward.restype = ctypes.c_int
    L.irsde_comm_unique_id.argtypes = [vp]
    L.irsde_comm_unique_id.restype = ctypes.c_int
    L.irsde_comm_init.argtypes = [vp, vp, i32, i32]
    L.irsde_comm_init.restype = ctypes.c_int
    L.irsde_broadcast_weights.argtypes = [vp, i32, vp]
    L.irsde_broadcast_weights.restype = ctypes.c_int
    L.irsde_gather.argtypes = [vp, vp, vp, ctypes.POINTER(i64), vp]
    L.irsde_gather.restype = ctypes.c_int
    L.irsde_random_states.argtypes = [vp, vp, vp, vp, vp, vp, i32, i64, vp]
    L.irsde_random_states.restype = ctypes.c_int
    L.irsde_set_lens.argtypes = [vp, fp, i32, vp]
    L.irsde_set_lens.restype = ctypes.c_int
    L.irsde_trim.argtypes = [vp]
    L.irsde_trim.restype = ctypes.c_int
    L.irsde_profile_begin.argtypes = [vp]
    L.irsde_profile_begin.restype = ctypes.c_int
    L.irsde_profile_end.argtypes = [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double),
                                    ctypes.POINTER(i64), i32]
    L.irsde_profile_end.restype = ctypes.c_int
    L.irsde_profile_end_bytes.argtypes = [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double),
                                          ctypes.POINTER(i64), ctypes.POINTER(ctypes.c_double), i32]
    L.irsde_profile_end_bytes.restype = ctypes.c_int
    _lib = L
    return L


class IrsdeError(RuntimeError):
    pass


def check(rc, ctx=None):
    if rc != 0:
        msg = load().irsde_last_error(ctx)
        raise IrsdeError("irsde_b200 error %d: %s" % (rc, msg.decode() if msg else "?"))


def float_array(seq):
    arr = (ctypes.c_float * len(seq))(*[float(v) for v in seq])
    return arr


class Context:
    """Owns one ``irsde_ctx`` (one per model per device)."""

    def __init__(self, in_nc, out_nc, nf, depth, variant, precision, device_index, force_simt=False, ch_mult=None):
        L = load()
        cfg = Config(in_nc, out_nc, nf, depth, variant, precision, device_index, FLAG_FORCE_SIMT if force_simt else 0)
        h = ctypes.c_void_p()
        if ch_mult is not None:
            arr = (ctypes.c_int32 * len(ch_mult))(*ch_mult)
            check(L.irsde_create_ch_mult(ctypes.byref(cfg), arr, len(ch_mult), ctypes.byref(h)))
        else:
            check(L.irsde_create(ctypes.byref(cfg), ctypes.byref(h)))
        self.h = h
        self.L = L

    def close(self):
        if getattr(self, "h", None):
            self.L.irsde_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
