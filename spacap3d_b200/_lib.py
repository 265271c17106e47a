"""ctypes binding of libspacap3d_ops.so (include/spacap3d_ops.h).

There is deliberately NO fallback: if the CUDA library is missing or a call fails, an exception
is raised.  Nothing here imports the test oracle.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SPC_LIB_PATH lets a developer load an instrumented build of the same library (profiling only)
LIB_PATH = os.environ.get("SPC_LIB_PATH") or os.path.join(_HERE, "libspacap3d_ops.so")
ABI_VERSION = 20

_p = ctypes.c_void_p
_i = ctypes.c_int
_f = ctypes.c_float

# name -> argtypes, exactly the prototypes of include/spacap3d_ops.h
SIGNATURES = {
    "spc_furthest_point_sampling": [_p, _i, _i, _i, _p, _p, _p],
    "spc_furthest_point_sampling_ex": [_p, _i, _i, _i, _p, _p, _i, _p, ctypes.c_size_t, _p],
    "spc_furthest_point_sampling_ex2": [_p, _i, _i, _i, _p, _p, _i, _p, _p, _p, ctypes.c_size_t, _i, _p],
    "spc_gather_points": [_p, _p, _i, _i, _i, _i, _p, _p],
    "spc_gather_points_grad": [_p, _p, _i, _i, _i, _i, _p, _p],
    "spc_ball_query": [_p, _p, _i, _i, _i, _f, _i, _p, _p],
    "spc_ball_query_ex": [_p, _p, _i, _i, _i, _f, _i, _p, _p, ctypes.c_size_t, _p],
    "spc_group_points": [_p, _p, _i, _i, _i, _i, _i, _p, _p],
    "spc_group_points_grad": [_p, _p, _i, _i, _i, _i, _i, _p, _p],
    "spc_box_point_counts": [_p, _i, _p, _i, _i, _i, _p, _p],
    "spc_nms_boxes": [_p, _p, _p, _p, _i, _i, _i, _i, ctypes.c_double, _p, _p],
    "spc_scene_floor_height": [_p, _i, _i, _i, _f, _p, _p],
    "spc_prepare_point_clouds": [_p, _i, _p, _i, _p, _p, _p, _p, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                 _i, _i, _i, _i, _p, _p],
    "spc_vote_labels": [_p, _i, _p, _p, _p, _p, _i, _i, _i, ctypes.c_uint64, _p, _p, _p, _p, ctypes.c_size_t, _p],
    "spc_augment_boxes": [_p, _p, _i, _i, _p, _p],
    "spc_bn_relu_train_forward": [_p, _p, _p, _i, _i, _i, _f, _f, _p, _p, _p, _p, _p, _p, ctypes.c_size_t, _p],
    "spc_bn_relu_maxpool_train_forward": [_p, _p, _p, _i, _i, _i, _i, _f, _f, _p, _p, _p, _p, _p, _p, _p, _p,
                                          ctypes.c_size_t, _p],
    "spc_bn_relu_maxpool_train_backward": [_p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p, _p, _p, _p],
    "spc_bn_relu_train_backward": [_p, _p, _p, _p, _p, _p, _i, _i, _i, _p, _p, _p, _p, ctypes.c_size_t, _p],
    "spc_bn_relu_sync_stats": [_p, _i, _i, _i, _p, _p, ctypes.c_size_t, _p],
    "spc_bn_relu_sync_forward": [_p, _p, _p, _i, _i, _i, _i, _p, _f, _f, _p, _p, _p, _p, _p, _p],
    "spc_bn_relu_sync_backward_reduce": [_p, _p, _p, _p, _p, _p, _i, _i, _i, _p, _p, _p, _p, ctypes.c_size_t, _p],
    "spc_bn_relu_sync_backward": [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p, _p, _p, ctypes.c_size_t, _p],
    "spc_bn_relu_maxpool_sync_forward": [_p, _p, _p, _i, _i, _i, _i, _i, _p, _f, _f, _p, _p, _p, _p, _p, _p, _p, _p],
    "spc_bn_relu_maxpool_sync_backward_reduce": [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p, _p, _p, _p],
    "spc_bn_relu_maxpool_sync_backward": [_p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p, _p, _p,
                                          ctypes.c_size_t, _p],
    "spc_group_points_grad_ex": [_p, _p, _i, _i, _i, _i, _i, _p, _p, ctypes.c_size_t, _p],
    "spc_three_nn": [_p, _p, _i, _i, _i, _p, _p, _p],
    "spc_three_interpolate": [_p, _p, _p, _i, _i, _i, _i, _p, _p],
    "spc_three_interpolate_grad": [_p, _p, _p, _i, _i, _i, _i, _p, _p],
    "spc_three_nn_weights": [_p, _p, _i, _i, _i, _p, _p, _p],
    "spc_interp_cat_pm": [_p, _p, _p, _p, _i, _i, _i, _i, _i, _p, _p],
    "spc_pm_linear": [_p, _p, _i, _i, _p, _p, _p, _i, _i, _i, _p, _p, _p, _p, _p, _p, _i, _i, _p],
    "spc_sa_fused_forward": [_p, _p, _p, _p, _p, _p, _p, _i, _f, _p, _p, _p, _p,
                             _i, _i, _i, _i, _i, _i, _i, _p, _p, _p],
    "spc_sa_fused_forward_ex": [_p, _p, _p, _p, _p, _p, _p, _p, _p, _i, _f, _p, _p, _p, _p,
                                _i, _i, _i, _i, _i, _i, _i, _p, _p, _i, _p],
}
# bf16-storage twins (torch.autocast training): the same argument lists, the bf16 tensors passed as void pointers
BF16_TWINS = (
    "spc_group_points", "spc_group_points_grad", "spc_group_points_grad_ex",
    "spc_three_interpolate", "spc_three_interpolate_grad",
    "spc_bn_relu_train_forward", "spc_bn_relu_train_backward",
    "spc_bn_relu_maxpool_train_forward", "spc_bn_relu_maxpool_train_backward",
    "spc_bn_relu_sync_stats", "spc_bn_relu_sync_forward", "spc_bn_relu_sync_backward_reduce", "spc_bn_relu_sync_backward",
    "spc_bn_relu_maxpool_sync_forward", "spc_bn_relu_maxpool_sync_backward_reduce", "spc_bn_relu_maxpool_sync_backward",
)
SIGNATURES.update({name + "_bf16": SIGNATURES[name] for name in BF16_TWINS})

_lib = None


class SpcError(RuntimeError):
    pass


def load():
    """dlopen the library (once).  Raises if it has not been built: there is no CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SpcError(
            "libspacap3d_ops.so is not built (%s).  Run `python -m spacap3d_b200.build` "
            "(or __graft_entry__.build()).  There is no CPU / PyTorch fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    lib.spc_abi_version.restype = _i
    lib.spc_last_error.restype = ctypes.c_char_p
    if lib.spc_abi_version() != ABI_VERSION:
        raise SpcError("libspacap3d_ops.so ABI %d != expected %d; rebuild" %
                       (lib.spc_abi_version(), ABI_VERSION))
    lib.spc_ball_query_workspace_bytes.argtypes = [_i, _i]
    lib.spc_ball_query_workspace_bytes.restype = ctypes.c_size_t
    lib.spc_group_points_grad_workspace_bytes.argtypes = [_i, _i, _i, _i]
    lib.spc_group_points_grad_workspace_bytes.restype = ctypes.c_size_t
    lib.spc_bn_relu_workspace_bytes.argtypes = [_i]
    lib.spc_bn_relu_workspace_bytes.restype = ctypes.c_size_t
    lib.spc_vote_labels_workspace_bytes.argtypes = [_i, _i]
    lib.spc_vote_labels_workspace_bytes.restype = ctypes.c_size_t
    lib.spc_fps_workspace_bytes.argtypes = [_i, _i, _i]
    lib.spc_fps_workspace_bytes.restype = ctypes.c_size_t
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = _i
    _lib = lib
    return lib


UNSUPPORTED = 3


class SpcUnsupported(SpcError):
    """The library has no kernel for this shape (SPC_ERR_UNSUPPORTED); nothing was launched."""


def call(name, *args):
    lib = load()
    status = getattr(lib, name)(*args)
    if status == UNSUPPORTED:
        raise SpcUnsupported("%s: %s" % (name, lib.spc_last_error().decode("utf-8", "replace")))
    if status != 0:
        raise SpcError("%s failed (status %d): %s" %
                       (name, status, lib.spc_last_error().decode("utf-8", "replace")))
