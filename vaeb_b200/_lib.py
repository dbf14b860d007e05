"""ctypes binding of include/vaeb_b200.h.  There is no CPU fallback: if the CUDA library has
not been built the import of any compute entry point fails loudly."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvaeb_b200.so")

EST_LB, EST_LA, EST_FVB, EST_FVB_SAMPLED = 0, 1, 2, 3
VARIANT_VAEB, VARIANT_FULLBAYES = 0, 1
PREC_FP32, PREC_BF16, PREC_BF16X3 = 0, 1, 2

# buffers addressable through vaeb_{get,set}_tensors
BUF_PARAMS, BUF_ADA, BUF_GRADS, BUF_VMU, BUF_VSIG, BUF_ADA_MU, BUF_ADA_SIG, BUF_GMU, BUF_GSIG, BUF_ADA2 = range(10)
OPT_ADAGRAD, OPT_ADADELTA, OPT_ADAM = 0, 1, 2
BUF_ADAM_V = 9          # Adam's second moment (BUF_ADA is its first moment)
BUF_THETA, BUF_ZETA = 10, 11    # sampled full VB: theta and zeta of the next update
AE_DEGENERATE, AE_VANILLA = 0, 1


class Config(C.Structure):
    _fields_ = [("input_dim", C.c_int32), ("hidden_units", C.c_int32), ("latent_size", C.c_int32),
                ("batch_size", C.c_int32), ("L", C.c_int32), ("continuous", C.c_int32),
                ("estimator", C.c_int32), ("variant", C.c_int32), ("precision", C.c_int32),
                ("device", C.c_int32), ("learning_rate", C.c_float), ("adagrad_eps", C.c_float),
                ("prior_scale", C.c_float), ("sigma_vb_init", C.c_float), ("seed", C.c_uint64),
                ("encoder_hidden_layers", C.c_int32), ("reserved0", C.c_int32)]


EXPORTS = {
    # name: (restype, argtypes)
    "vaeb_last_error": (C.c_char_p, []),
    "vaeb_version": (C.c_int, []),
    "vaeb_config_size": (C.c_int, []),
    "vaeb_create": (C.c_int, [C.POINTER(Config), C.POINTER(C.c_void_p)]),
    "vaeb_destroy": (C.c_int, [C.c_void_p]),
    "vaeb_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "vaeb_synchronize": (C.c_int, [C.c_void_p]),
    "vaeb_num_tensors": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int64)]),
    "vaeb_tensor_shape": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "vaeb_set_tensors": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_void_p)]),
    "vaeb_get_tensors": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_void_p)]),
    "vaeb_device_buffer": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "vaeb_upload_data": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "vaeb_update": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.POINTER(C.c_float)]),
    "vaeb_update_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.POINTER(C.c_float)]),
    "vaeb_update_many": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "vaeb_update_host_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "vaeb_update_host_async_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_float]),
    "vaeb_diag_tile_schedule": (C.c_int, [C.c_int32] * 6 + [C.c_void_p] * 3),
    "vaeb_set_optimizer": (C.c_int, [C.c_void_p, C.c_int32, C.c_float]),
    "vaeb_set_adam": (C.c_int, [C.c_void_p, C.c_float, C.c_float, C.c_float]),
    "vaeb_adam_step": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "vaeb_set_adam_step": (C.c_int, [C.c_void_p, C.c_int64]),
    "vaeb_set_kl_weight": (C.c_int, [C.c_void_p, C.c_float, C.c_int64]),
    "vaeb_kl_step": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "vaeb_set_kl_step": (C.c_int, [C.c_void_p, C.c_int64]),
    "vaeb_ae_train": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.POINTER(C.c_float)]),
    "vaeb_ae_forward": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]),
    "vaeb_collect": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.c_void_p]),
    "vaeb_validate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.POINTER(C.c_float), C.c_void_p]),
    "vaeb_gradients": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p,
                                 C.POINTER(C.c_float), C.c_void_p]),
    "vaeb_apply_update": (C.c_int, [C.c_void_p]),
    "vaeb_is_logpx": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int64,
                                C.c_void_p, C.c_void_p]),
    "vaeb_reconstruct": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "vaeb_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "vaeb_encode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "vaeb_sample": (C.c_int, [C.c_void_p, C.c_int64, C.c_uint32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                              C.c_void_p]),
    "vaeb_validate_terms": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "vaeb_mlp_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.POINTER(C.c_int32),
                                   C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int32, C.c_void_p]),
    "vaeb_philox_normal": (C.c_int, [C.c_void_p, C.c_int32, C.c_uint32, C.c_uint32, C.c_int64, C.c_int64, C.c_void_p]),
    "vaeb_set_step_counter": (C.c_int, [C.c_void_p, C.c_uint32]),
    "vaeb_step_counter": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint32)]),
    "vaeb_comm_unique_id": (C.c_int, [C.c_char_p, C.c_void_p]),
    "vaeb_comm_attach": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int32, C.c_int32]),
    "vaeb_comm_detach": (C.c_int, [C.c_void_p]),
    "vaeb_set_hidden_activation": (C.c_int, [C.c_void_p, C.c_int32]),
    "vaeb_comm_p2p_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "vaeb_comm_p2p_attach": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32]),
    "vaeb_profile_update": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p]),
    "vaeb_profile_optimizer": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_double)]),
    "vaeb_tc_gemm_test": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                    C.c_void_p, C.c_void_p, C.c_void_p]),
    "vaeb_launch_count": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "vaeb_step_kernel": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(C.c_int32)]),
    "vaeb_host_alloc": (C.c_int, [C.c_int64, C.POINTER(C.c_void_p)]),
    "vaeb_host_free": (C.c_int, [C.c_void_p]),
}

_lib = None


def load():
    """dlopen the in-tree library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "vaeb_b200: %s is missing. Build it with `python -m vaeb_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)       # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    if lib.vaeb_config_size() != C.sizeof(Config):
        raise RuntimeError("vaeb_b200: %s was built from another include/vaeb_b200.h (struct vaeb_config is %d bytes there, "
                           "%d here): rebuild it with `python -m vaeb_b200.build`"
                           % (LIB_PATH, lib.vaeb_config_size(), C.sizeof(Config)))
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().vaeb_last_error().decode("utf-8", "replace")
        if rc == 1:
            raise ValueError("vaeb_b200: " + msg)
        raise RuntimeError("vaeb_b200 (code %d): %s" % (rc, msg))


def nccl_library_path():
    """The libnccl.so.2 torch bundles (falls back to the system one)."""
    try:
        import nvidia.nccl as _n  # namespace package
        for p in list(getattr(_n, "__path__", [])):
            cand = os.path.join(p, "lib", "libnccl.so.2")
            if os.path.exists(cand):
                return cand
    except Exception:
        pass
    return "libnccl.so.2"
