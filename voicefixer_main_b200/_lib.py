"""ctypes binding of libb200vf.so (C ABI in include/b200vf.h).

There is no fallback: if the shared library has not been built (python __graft_entry__.py build, or
make -C voicefixer_main_b200/csrc) importing the engine raises, and without a CUDA device vf_create fails
with VF_ENODEVICE.  Nothing here computes on the data path; it only marshals pointers.
"""
import ctypes
import os
from ctypes import (POINTER, Structure, byref, c_char_p, c_double, c_float, c_int, c_int64, c_size_t, c_uint, c_void_p)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200vf.so")

VF_OK, VF_EINVAL, VF_ENODEVICE, VF_ECUDA, VF_ESTATE, VF_EDEVICE, VF_EASSERT = 0, -1, -2, -3, -4, -5, -6

EXPORTS = [
    "vf_default_config", "vf_create", "vf_destroy", "vf_last_error", "vf_load_weights", "vf_frontend",
    "vf_unet_mel", "vf_vocoder", "vf_vocoder_out_len", "vf_restore", "vf_restore_host", "vf_restore_stages",
    "vf_to_log", "vf_from_log", "vf_to_pcm16", "vf_workspace_bytes", "vf_check_errors", "vf_set_option", "vf_launch_count",
    "vf_enable_stage_timing", "vf_stage_times", "vf_selftest_gemm", "vf_enable_op_timing", "vf_op_count", "vf_op_info",
    "vf_restore_ex", "vf_ssr_forward", "vf_ssr_restore", "vf_ssr_restore_host", "vf_ssr_unet", "vf_ssr_stages", "vf_istft",
    "vf_mel", "vf_finalize", "vf_plan_cache_info", "vf_resample_poly", "vf_lsd", "vf_sispec", "vf_to_pcm16_ex", "vf_amp_to_original_f",
    "vf_restore_varlen", "vf_ssr_restore_varlen",
]
VF_RESTORE_UNIFY_ENERGY = 1


class VfConfig(Structure):
    _fields_ = [("sample_rate", c_int), ("n_fft", c_int), ("hop", c_int), ("n_mels", c_int),
                ("voc_cond_channels", c_int), ("voc_cond_layers", c_int), ("voc_channels", c_int),
                ("voc_num_stages", c_int), ("voc_scales", c_int * 8), ("voc_depth", c_int * 8),
                ("voc_stage_slope", c_float), ("voc_res_slope", c_float), ("voc_min_db", c_float),
                ("voc_ref_db", c_float), ("voc_amp_floor", c_float), ("voc_tail_value", c_float),
                ("voc_tail_base", c_int), ("voc_mel_weight_a", c_double), ("voc_mel_weight_b", c_double),
                ("voc_tail_tanh", c_int)]


class VfTensorDesc(Structure):
    _fields_ = [("name", c_char_p), ("data", c_void_p), ("ndim", c_int), ("shape", c_int64 * 4),
                ("on_device", c_int)]


class EngineError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libb200vf error {code}: {msg}")
        self.code = code


_lib = None


def load_library():
    """Load libb200vf.so or raise: the product has no CPU / PyTorch fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build the CUDA extension first "
            "(python -c 'import __graft_entry__ as g; g.build()' or make -C voicefixer_main_b200/csrc). "
            "voicefixer_main_b200 has no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    P = c_void_p
    lib.vf_default_config.argtypes = [POINTER(VfConfig)]
    lib.vf_default_config.restype = None
    lib.vf_create.argtypes = [POINTER(P), c_int, POINTER(VfConfig)]
    lib.vf_destroy.argtypes = [P]
    lib.vf_destroy.restype = None
    lib.vf_last_error.argtypes = [P]
    lib.vf_last_error.restype = c_char_p
    lib.vf_load_weights.argtypes = [P, POINTER(VfTensorDesc), c_int]
    lib.vf_frontend.argtypes = [P, P, c_int, c_int64, P, P, P, P, P]
    lib.vf_unet_mel.argtypes = [P, P, c_int, c_int, P, P]
    lib.vf_vocoder.argtypes = [P, P, c_int, c_int, P, P]
    lib.vf_vocoder_out_len.argtypes = [P, c_int]
    lib.vf_vocoder_out_len.restype = c_int64
    lib.vf_restore.argtypes = [P, P, c_int, c_int64, P, P]
    lib.vf_restore_host.argtypes = [P, P, c_int, c_int64, P, P]
    lib.vf_restore_stages.argtypes = [P, c_int, c_int64, P, P, P]
    lib.vf_to_log.argtypes = [P, P, P, c_int64, P]
    lib.vf_from_log.argtypes = [P, P, P, c_int64, P]
    lib.vf_to_pcm16.argtypes = [P, P, P, c_int64, P]
    lib.vf_workspace_bytes.argtypes = [P, c_int, c_int64, POINTER(c_size_t)]
    lib.vf_check_errors.argtypes = [P, P]
    lib.vf_set_option.argtypes = [P, c_char_p, c_int]
    lib.vf_launch_count.argtypes = [P]
    lib.vf_launch_count.restype = c_int64
    lib.vf_enable_stage_timing.argtypes = [P, c_int]
    lib.vf_stage_times.argtypes = [P, POINTER(c_float * 4)]
    lib.vf_selftest_gemm.argtypes = [P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, POINTER(c_double),
                                     POINTER(c_double)]
    lib.vf_enable_op_timing.argtypes = [P, c_int]
    lib.vf_op_count.argtypes = [P]
    lib.vf_op_info.argtypes = [P, c_int, POINTER(c_float), POINTER(c_double), POINTER(c_double), POINTER(c_int),
                               POINTER(c_int), POINTER(c_int), c_char_p, c_int, POINTER(c_double)]
    lib.vf_restore_ex.argtypes = [P, P, c_int, c_int64, P, c_uint, P]
    lib.vf_restore_varlen.argtypes = [P, P, c_int, c_int64, POINTER(c_int64), P, c_uint, P]
    lib.vf_ssr_forward.argtypes = [P, P, P, c_int, c_int64, P, P]
    lib.vf_ssr_restore.argtypes = [P, P, c_int, c_int64, P, P]
    lib.vf_ssr_restore_host.argtypes = [P, P, c_int, c_int64, P, P]
    lib.vf_ssr_restore_varlen.argtypes = [P, P, c_int, c_int64, POINTER(c_int64), P, P]
    lib.vf_ssr_unet.argtypes = [P, P, c_int, c_int, P, P]
    lib.vf_ssr_stages.argtypes = [P, c_int, c_int64, P, P, P]
    lib.vf_istft.argtypes = [P, P, P, c_int, c_int, c_int64, P, P]
    lib.vf_mel.argtypes = [P, P, c_int64, c_int64, c_int64, c_int64, c_int64, P, P]
    lib.vf_finalize.argtypes = [P, P, c_int, c_int64, c_int64, P, P]
    lib.vf_plan_cache_info.argtypes = [P, POINTER(c_int), POINTER(c_size_t), POINTER(c_size_t), POINTER(c_int64)]
    lib.vf_resample_poly.argtypes = [P, P, c_int, c_int64, c_int, c_int, P, c_int, P, c_int64, P]
    lib.vf_to_pcm16_ex.argtypes = [P, P, P, c_int64, c_int, P]
    lib.vf_amp_to_original_f.argtypes = [P, P, P, c_int, c_int, P, P]
    lib.vf_lsd.argtypes = [P, P, P, c_int, c_int, c_int, P, P]
    lib.vf_sispec.argtypes = [P, P, P, c_int, c_int64, c_int, c_int, P, P]
    _lib = lib
    return lib


def check(lib, ctx, rc):
    if rc != VF_OK:
        msg = lib.vf_last_error(ctx)
        raise EngineError(rc, msg.decode() if msg else "")
    return rc
