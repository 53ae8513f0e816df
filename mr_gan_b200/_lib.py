"""ctypes binding of libmrgan.so (include/mrgan.h).

There is no CPU fallback: if the library is missing it is built with nvcc, and if
that fails -- or if a compute entry point is called without a Blackwell GPU -- the
call raises.  Nothing in this package ever routes through ``oracle/``.
"""
import ctypes as C
import os

from . import build as _build

_LIB = None


class Config(C.Structure):
    _fields_ = [("model", C.c_int), ("n_folds", C.c_int), ("batch", C.c_int), ("n_classes", C.c_int),
                ("noise_dim", C.c_int), ("precision", C.c_int), ("shared_t", C.c_int),
                ("eval_each_epoch", C.c_int), ("device", C.c_int),
                ("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("adam_eps", C.c_float),
                ("bn_eps", C.c_float), ("unlabeled_weight", C.c_float),
                ("sigma_in", C.c_float), ("sigma_hidden", C.c_float),
                ("hidden_act", C.c_int), ("leaky_alpha", C.c_float), ("dropout", C.c_float)]


class FoldShape(C.Structure):
    _fields_ = [("D", C.c_int), ("n_train", C.c_int), ("n_test", C.c_int), ("seed", C.c_uint64)]


class EpochStats(C.Structure):
    _fields_ = [("loss_lab", C.c_float), ("loss_unl", C.c_float), ("train_err", C.c_float),
                ("loss_gen", C.c_float), ("test_err", C.c_float)]


_fp = C.POINTER(C.c_float)
_ip = C.POINTER(C.c_int32)
_H = C.c_void_p

# every symbol include/mrgan.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "mrgan_default_config": (C.c_int, [C.c_int, C.POINTER(Config)]),
    "mrgan_create": (C.c_int, [C.POINTER(Config), C.POINTER(FoldShape), C.POINTER(_H)]),
    "mrgan_destroy": (C.c_int, [_H]),
    "mrgan_last_error": (C.c_char_p, [_H]),
    "mrgan_sync": (C.c_int, [_H]),
    "mrgan_num_params": (C.c_int64, [_H, C.c_int, C.c_int]),
    "mrgan_set_params": (C.c_int, [_H, C.c_int, C.c_int, _fp, C.c_int64]),
    "mrgan_get_params": (C.c_int, [_H, C.c_int, C.c_int, _fp, C.c_int64]),
    "mrgan_get_adam": (C.c_int, [_H, C.c_int, C.c_int, _fp, _fp, C.c_int64]),
    "mrgan_get_counters": (C.c_int, [_H, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "mrgan_load_fold": (C.c_int, [_H, C.c_int, _fp, _ip, _fp, _ip]),
    "mrgan_load_dataset": (C.c_int, [_H, C.c_int, _fp, _ip, C.c_int, C.c_int]),
    "mrgan_prepare_fold": (C.c_int, [_H, C.c_int, C.c_int, _ip, _ip]),
    "mrgan_disc_step": (C.c_int, [_H, C.c_int, _fp, _ip, _fp, _fp, _fp]),
    "mrgan_gen_step": (C.c_int, [_H, C.c_int, _fp, _fp, _fp]),
    "mrgan_test_batch": (C.c_int, [_H, C.c_int, _fp, _ip, C.c_int, _fp]),
    "mrgan_train_epoch": (C.c_int, [_H, _ip, _ip, _ip, C.POINTER(EpochStats)]),
    "mrgan_epoch_result": (C.c_int, [_H, C.POINTER(EpochStats)]),
    "mrgan_set_epoch_rows": (C.c_int, [_H, C.c_int, _ip, C.c_int, _ip, C.c_int]),
    "mrgan_train_epoch_seeded": (C.c_int, [_H, C.c_uint32, C.POINTER(EpochStats)]),
    "mrgan_debug_epoch_indices": (C.c_int, [_H, C.c_int, _ip]),
    "mrgan_eval": (C.c_int, [_H, C.c_int, _fp]),
    "mrgan_nccl_unique_id": (C.c_int, [C.c_void_p]),
    "mrgan_dp_init": (C.c_int, [_H, C.c_int, C.c_int, C.c_void_p]),
    "mrgan_dp_init_virtual": (C.c_int, [_H, C.c_int]),
    "mrgan_dp_ipc_export": (C.c_int, [_H, C.c_void_p]),
    "mrgan_dp_ipc_open": (C.c_int, [_H, C.c_void_p, C.c_int]),
    "mrnn_step": (C.c_int, [_H, C.c_int, _fp, _ip, C.c_int, _fp]),
    "mrnn_train_epoch": (C.c_int, [_H, _ip, C.c_int, _fp]),
    "mrnn_evaluate": (C.c_int, [_H, C.c_int, _fp]),
    "mrgan_svm_fit": (C.c_int, [_H, _ip, C.c_int, C.c_float, _fp, C.c_float, _ip]),
    "mrgan_svm_fit_folds": (C.c_int, [_H, _ip, C.c_int, _fp, _fp, C.c_float, _ip]),
    "mrgan_svm_cv": (C.c_int, [_H, _ip, C.c_int, _ip, C.c_int, _fp, C.c_int, _fp, C.c_int, C.c_float, _ip]),
    "mrgan_svm_eval": (C.c_int, [_H, C.c_int, _fp]),
    "mrgan_svm_decision": (C.c_int, [_H, C.c_int, _fp]),
    "mrgan_predict": (C.c_int, [_H, C.c_int, _ip, _fp]),
    "mrgan_predict_rows": (C.c_int, [_H, C.c_int, _fp, C.c_int, _ip, _fp]),
    "mrgan_confusion": (C.c_int, [_H, _ip]),
    "mrgan_input_grad": (C.c_int, [_H, C.c_int, _fp, C.c_int, _ip, _fp]),
    "mrgan_saliency": (C.c_int, [_H, _fp]),
    "mrgan_fill_normal": (C.c_int, [_H, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _fp]),
    "mrgan_adam_flat": (C.c_int, [_H, _fp, _fp, _fp, _fp, C.c_int64, C.c_int]),
    "mrgan_time_op": (C.c_int, [_H, C.c_int, C.c_int, _fp]),
    "mrgan_debug_buffer": (C.c_int, [_H, C.c_int, C.c_int, _fp, C.c_int, C.c_int]),
    "mrgan_debug_gemm": (C.c_int, [_H, C.c_int, C.c_int, C.c_int, C.c_int, _fp, _fp, _fp, C.c_int]),
    "mrgan_debug_gemm_time": (C.c_int, [_H, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _fp]),
    "mrgan_kernel_launches": (C.c_int64, [_H]),
    "mrgan_last_device_ms": (C.c_double, [_H]),
    "mrgan_version": (C.c_char_p, []),
    "mrgan_abi_info": (C.c_int, [C.POINTER(C.c_int)]),
}

ABI_VERSION = 3      # MRGAN_ABI_VERSION of include/mrgan.h this binding was written against


def lib_path():
    return _build.LIB


def load():
    """Load (building if needed) libmrgan.so and declare every prototype.  Raises on failure."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = os.environ.get("MRGAN_LIB")                    # MRGAN_LIB: a prebuilt library (kernel A/B experiments)
    if path:
        if not os.path.exists(path):
            raise RuntimeError("MRGAN_LIB=%s does not exist" % path)
    else:
        path = _build.build()        # no-op when the library matches the sources (content hash); rebuilds a stale one
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the library lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    # the structs above are laid out by hand: refuse a library whose ABI differs instead of corrupting memory
    info = (C.c_int * 4)()
    if lib.mrgan_abi_info(info) != 0:
        raise RuntimeError("mrgan_abi_info failed")
    want = [ABI_VERSION, C.sizeof(Config), C.sizeof(FoldShape), C.sizeof(EpochStats)]
    if list(info) != want:
        raise RuntimeError("libmrgan.so ABI mismatch: library %s, binding %s (version, sizeof config / fold_shape / "
                           "epoch_stats)" % (list(info), want))
    _LIB = lib
    return lib


def fptr(a):
    return a.ctypes.data_as(_fp)


def iptr(a):
    return a.ctypes.data_as(_ip)
