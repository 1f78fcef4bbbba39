"""ctypes binding of libddn_b200.so (the C ABI declared in include/ddn_b200.h).

There is no CPU or PyTorch fallback: if the library cannot be loaded, importing this module raises.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libddn_b200.so")

PRECISION_FP32_SIMT, PRECISION_BF16X3, PRECISION_BF16 = 0, 1, 2
MODE_INFER, MODE_TRAIN, MODE_EVAL_SAVE = 0, 1, 2
GRAD_BUCKET_FN = ctypes.CFUNCTYPE(None, ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_int64)
TERM_MATCH, TERM_HINGE, TERM_HINGE_INV = 0, 1, 2
TERM_PIXEL_WEIGHT = 1
MAX_TERMS = 8

c_f32p = ctypes.POINTER(ctypes.c_float)
vp, i32, i64, f32, sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_size_t


class TensorEntry(ctypes.Structure):
    _fields_ = [("name", ctypes.c_char * 64), ("ndim", ctypes.c_int32), ("shape", ctypes.c_int32 * 4),
                ("offset", ctypes.c_int64), ("numel", ctypes.c_int64)]


class LossTerm(ctypes.Structure):
    _fields_ = [("idx_a", vp), ("idx_b", vp), ("gt_b", vp), ("n", i64), ("n_gt", i64),
                ("kind", ctypes.c_int32), ("flags", ctypes.c_int32), ("margin", f32), ("m_pixel", f32),
                ("len", vp), ("len_gt", vp)]


class ProfileEntry(ctypes.Structure):
    _fields_ = [("name", ctypes.c_char * 32), ("launches", ctypes.c_int64), ("ms", ctypes.c_double), ("work", ctypes.c_double)]


class WithinSceneCfg(ctypes.Structure):
    _fields_ = [("match_loss_weight", f32), ("non_match_loss_weight", f32),
                ("scale_by_hard_negatives", ctypes.c_int32), ("has_blind", ctypes.c_int32),
                ("n_match", i64), ("n_masked", i64), ("n_background", i64), ("n_blind", i64),
                ("len_match", vp), ("len_masked", vp), ("len_background", vp), ("len_blind", vp)]


_SIGNATURES = {
    "ddn_abi_version": (i32, []),
    "ddn_last_error": (ctypes.c_char_p, []),
    "ddn_kernel_launch_count": (i64, []),
    "ddn_resnet34_8s_param_table": (i32, [i32, ctypes.POINTER(TensorEntry), i32]),
    "ddn_resnet34_8s_buffer_table": (i32, [ctypes.POINTER(TensorEntry), i32]),
    "ddn_resnet34_8s_param_count": (i64, [i32]),
    "ddn_resnet34_8s_buffer_count": (i64, []),
    "ddn_resnet34_8s_workspace_bytes": (sz, [i32, i32, i32, i32, i32, i32]),
    "ddn_resnet34_8s_weight_cache_bytes": (sz, [i32]),
    "ddn_resnet34_8s_set_weight_cache": (i32, [vp, sz, vp, ctypes.c_uint64, i32]),
    "ddn_resnet34_8s_forward": (i32, [vp, vp, vp, vp, vp, sz, i32, i32, i32, i32, i32, i32, f32, f32, i32, vp, vp]),
    "ddn_resnet34_8s_backward": (i32, [vp, vp, vp, vp, vp, sz, i32, i32, i32, i32, i32, i32, f32, i32, GRAD_BUCKET_FN, vp, vp]),
    "ddn_contrastive_terms_forward_lowres": (i32, [vp, vp, i32, i32, i32, i32, i32, i32, ctypes.POINTER(LossTerm), i32, vp, vp, vp]),
    "ddn_contrastive_terms_backward_lowres": (i32, [vp, vp, i32, i32, i32, i32, i32, i32, ctypes.POINTER(LossTerm), i32,
                                                    vp, vp, vp, vp, vp]),
    "ddn_resnet34_8s_grad_buckets": (i32, [i32, ctypes.POINTER(i64), i32]),
    "ddn_contrastive_terms_forward": (i32, [vp, vp, i64, i64, i64, i32, i64, i32, i32, ctypes.POINTER(LossTerm), i32, vp, vp, vp]),
    "ddn_contrastive_terms_backward": (i32, [vp, vp, i64, i64, i64, i32, i64, i32, i32, ctypes.POINTER(LossTerm), i32,
                                             vp, vp, vp, vp, vp]),
    "ddn_within_scene_compose": (i32, [vp, vp, i32, i32, ctypes.POINTER(WithinSceneCfg), vp, vp, vp]),
    "ddn_within_scene_loss_host": (i32, [vp, vp, i32, i32, i32, i32, vp, vp, i64, vp, vp, i64, vp, vp, i64,
                                         f32, f32, f32, f32, i32, vp]),
    "ddn_conv2d_workspace_bytes": (sz, [i32] * 10),
    "ddn_conv2d_forward": (i32, [vp, vp, vp] + [i32] * 10 + [vp, sz, vp]),
    "ddn_conv2d_backward": (i32, [vp, vp, vp, vp, vp] + [i32] * 10 + [vp, sz, vp]),
    "ddn_batchnorm_workspace_bytes": (sz, [i64, i32]),
    "ddn_batchnorm_forward": (i32, [vp] * 9 + [i64, i32, i32, i32, f32, f32, vp, sz, vp]),
    "ddn_batchnorm_backward": (i32, [vp] * 10 + [i64, i32, i32, vp, sz, vp]),
    "ddn_upsample_bilinear_forward": (i32, [vp, vp, i32, i32, i32, i32, i32, vp]),
    "ddn_upsample_bilinear_backward": (i32, [vp, vp, i32, i32, i32, i32, i32, vp]),
    "ddn_scale_inplace": (i32, [vp, i64, f32, vp]),
    "ddn_sample_non_matches_scratch_bytes": (sz, [i32, i32]),
    "ddn_sample_non_matches": (i32, [vp, i32, i32, vp, vp, i64, vp, i64, vp, vp, vp, sz, vp]),
    "ddn_find_pixel_correspondences_scratch_bytes": (sz, [i64]),
    "ddn_find_pixel_correspondences": (i32, [vp, vp, i32, i32, vp, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]),
    "ddn_find_best_match": (i32, [vp, i64, i64, i32, i32, i32, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp]),
    "ddn_adam_step": (i32, [vp, vp, vp, vp, i64, i64, f32, f32, f32, f32, f32, f32, vp]),
    "ddn_profile_enable": (i32, [i32]),
    "ddn_profile_reset": (i32, []),
    "ddn_profile_read": (i32, [ctypes.POINTER(ProfileEntry), i32]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def _load():
    if not os.path.exists(LIB_PATH):
        # fresh checkout: compile the library in-tree (nvcc cross-compiles sm_100a without a GPU).  Still no fallback: if
        # nvcc is not there either, importing the package fails.
        try:
            import importlib.util
            spec = importlib.util.spec_from_file_location("_ddn_build", os.path.join(_HERE, "build.py"))
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
            mod.build()
        except Exception as e:
            raise ImportError(
                "libddn_b200.so is missing at %s and building it failed (%s): run `python "
                "pytorch-dense-correspondence_b200/build.py`.  There is no fallback path." % (LIB_PATH, e))
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError here == header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.ddn_abi_version() != 3:
        raise ImportError("libddn_b200.so ABI version mismatch")
    return lib


lib = _load()


class DdnError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        raise DdnError("libddn_b200 error %d: %s" % (rc, lib.ddn_last_error().decode()))


def ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda_f32(t, name, contiguous=True):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor: this path has no CPU fallback" % name)
    if t.dtype != torch.float32:
        raise RuntimeError("%s must be float32 (got %s)" % (name, t.dtype))
    if contiguous and not t.is_contiguous():
        raise RuntimeError("%s must be contiguous" % name)


def param_table(D):
    n = lib.ddn_resnet34_8s_param_table(D, None, 0)
    arr = (TensorEntry * n)()
    lib.ddn_resnet34_8s_param_table(D, arr, n)
    return [(e.name.decode(), tuple(e.shape[:e.ndim]), int(e.offset), int(e.numel)) for e in arr]


def buffer_table():
    n = lib.ddn_resnet34_8s_buffer_table(None, 0)
    arr = (TensorEntry * n)()
    lib.ddn_resnet34_8s_buffer_table(arr, n)
    return [(e.name.decode(), tuple(e.shape[:e.ndim]), int(e.offset), int(e.numel)) for e in arr]


def grad_buckets(D):
    """[(offset, numel)] of the 4 gradient buckets in the order the backward completes them (last layers first)."""
    arr = (i64 * 5)()
    n = lib.ddn_resnet34_8s_grad_buckets(D, arr, 5)
    ends = [int(arr[4])] + [int(arr[i]) for i in range(n - 1)]
    return [(int(arr[i]), ends[i] - int(arr[i])) for i in range(n)]


NO_BUCKET_CALLBACK = ctypes.cast(None, GRAD_BUCKET_FN)


def profile_read():
    """{class name: {"launches", "ms", "flops" (conv_*) or "bytes" (loss_*)}} for the kernels timed since the last reset."""
    arr = (ProfileEntry * 16)()
    n = lib.ddn_profile_read(arr, 16)
    out = {}
    for e in arr[:n]:
        name = e.name.decode()
        out[name] = {"launches": int(e.launches), "ms": float(e.ms), ("flops" if name.startswith("conv") else "bytes"): float(e.work)}
    return out


def launch_count():
    return int(lib.ddn_kernel_launch_count())
