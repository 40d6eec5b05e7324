"""ctypes binding of libb200mdm.so (C ABI declared in include/b200mdm.h).

There is deliberately no fallback: if the shared library is missing, or a call fails, this raises.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200MDM_LIB") or os.path.join(HERE, "lib", "libb200mdm.so")   # (override: A/B builds of the same ABI)

OK, EINVAL, ECUDA, ESTATE, ENOTIMPL = 0, -1, -2, -3, -4
ARCH = {"trans_enc": 0, "trans_dec": 1}
COND_NONE, COND_TEXT, COND_ACTION = 0, 1, 2
MODE_X0, MODE_DDPM, MODE_DDIM = 0, 1, 2
TARGET = {None: 0, "single": 1, "multi": 2, "split": 3}
FLAG_CONST_NOISE, FLAG_CLIP_DENOISED, FLAG_PHILOX_NOISE = 1, 2, 4
SCHED_STRIDE = 8

# every symbol include/b200mdm.h declares (tests check that the library exports all of them)
SYMBOLS = [
    "b200mdm_last_error", "b200mdm_version", "b200mdm_create", "b200mdm_destroy", "b200mdm_load_weight",
    "b200mdm_finalize_weights", "b200mdm_set_schedule", "b200mdm_set_cond", "b200mdm_set_cond_dec", "b200mdm_set_prefix",
    "b200mdm_set_inpaint", "b200mdm_set_target",
    "b200mdm_denoise", "b200mdm_sample_step", "b200mdm_sample_loop", "b200mdm_q_sample", "b200mdm_launch_count",
    "b200mdm_sample_loop_range", "b200mdm_set_noise_stream", "b200mdm_philox_normal",
    "b200mdm_recover_from_ric", "b200mdm_test_gemm_f16", "b200mdm_test_attention", "b200mdm_test_cross_attention", "b200mdm_test_qkv_attention", "b200mdm_test_gemm_resid_ln",
    "b200mdm_test_gemm2_plan",
]


class Config(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in (
        "arch", "latent_dim", "ff_size", "num_layers", "num_heads", "njoints", "nfeats", "cond_mode", "cond_dim",
        "num_actions", "mask_frames", "pos_embed_max_len", "temb_rows", "context_len", "target_encoder", "n_goal_rows",
        "target_enc_layers")] + [("reserved", ctypes.c_int32 * 3)]


class B200MDMError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libb200mdm error %d: %s" % (code, msg))
        self.code = code


_lib = None


def load():
    """dlopen the engine.  torch must already be imported (shares its CUDA runtime)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libb200mdm.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'`; "
            "there is no CPU / PyTorch fallback for the sampling path." % LIB_PATH)
    import torch  # noqa: F401  (loads libcudart into the process before our library resolves it)
    lib = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
    vp, i32, i64, f32 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_float
    lib.b200mdm_last_error.restype = ctypes.c_char_p
    lib.b200mdm_last_error.argtypes = []
    lib.b200mdm_version.restype = i32
    lib.b200mdm_create.argtypes = [ctypes.POINTER(Config), ctypes.POINTER(vp)]
    lib.b200mdm_destroy.argtypes = [vp]
    lib.b200mdm_load_weight.argtypes = [vp, ctypes.c_char_p, vp, ctypes.POINTER(i64), i32]
    lib.b200mdm_finalize_weights.argtypes = [vp, vp]
    lib.b200mdm_set_schedule.argtypes = [vp, i32, vp, vp]
    lib.b200mdm_set_cond.argtypes = [vp, i32, i32, vp, vp, vp, i32, vp, vp]
    lib.b200mdm_set_cond_dec.argtypes = [vp, i32, i32, vp, vp, i32, vp, vp, i32, vp]
    lib.b200mdm_set_prefix.argtypes = [vp, vp, vp]
    if hasattr(lib, "b200mdm_set_target"):           # (absent from A/B builds that predate target conditioning)
        lib.b200mdm_set_target.argtypes = [vp, i32, vp, vp, vp]
    lib.b200mdm_set_inpaint.argtypes = [vp, vp, vp]
    lib.b200mdm_recover_from_ric.argtypes = [vp, i64, i64, i64, vp, vp, vp, i64, i64, i64, i32, i32, i32, vp]
    lib.b200mdm_denoise.argtypes = [vp, vp, vp, vp, vp]
    lib.b200mdm_sample_step.argtypes = [vp, i32, i32, vp, vp, i32, vp, vp, vp]
    lib.b200mdm_sample_loop.argtypes = [vp, i32, i32, vp, vp, vp, i64, i32, i32, vp]
    lib.b200mdm_sample_loop_range.argtypes = [vp, i32, i32, i32, vp, vp, vp, i64, i32, i32, vp]
    lib.b200mdm_set_noise_stream.argtypes = [vp, ctypes.c_uint64, i64]
    lib.b200mdm_philox_normal.argtypes = [vp, i32, i64, ctypes.c_uint64, i64, i32, vp]
    lib.b200mdm_q_sample.argtypes = [vp, f32, f32, vp, vp, vp, i64, vp]
    lib.b200mdm_launch_count.argtypes = [vp, i32]
    lib.b200mdm_launch_count.restype = i64
    lib.b200mdm_test_gemm_f16.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]
    lib.b200mdm_test_attention.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp]
    if hasattr(lib, "b200mdm_test_cross_attention"):
        lib.b200mdm_test_cross_attention.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, vp]
    lib.b200mdm_test_qkv_attention.argtypes = [vp, i32, vp, vp, vp, vp, i32, i32, vp]
    lib.b200mdm_test_gemm_resid_ln.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, vp]
    lib.b200mdm_test_gemm2_plan.argtypes = [i32, i32, i32, i32, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32)]
    for name in SYMBOLS:
        if not hasattr(lib, name) and os.environ.get("B200MDM_LIB"):
            continue                                  # an older A/B build of the same ABI may lack the newest test hooks
        fn = getattr(lib, name)
        if fn.restype is ctypes.c_int and name not in ("b200mdm_version",):
            fn.restype = i32
    _lib = lib
    return lib


def check(code):
    if code != OK:
        raise B200MDMError(code, load().b200mdm_last_error().decode("utf-8", "replace"))
