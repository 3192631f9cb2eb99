"""ctypes binding of libffb6d_b200.so (the C ABI declared in include/ffb6d_b200.h).

There is no CPU fallback: if the shared library is missing or fails to load,
importing this module raises, and every op in :mod:`ffb6d_b200.ops` fails with
it.  Build it with ``python -c "import __graft_entry__ as g; g.build()"`` or
``make -C ffb6d_b200/csrc``.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libffb6d_b200.so")

OK = 0
ERR_INVALID = -1
ERR_CUDA = -2
ERR_WORKSPACE = -3
ERR_NO_DEVICE = -4
LAYOUT_NCS = 0
LAYOUT_NSC = 1
MAX_K = 64


class FFB6DError(RuntimeError):
    """A libffb6d_b200 entry point returned a negative status."""

    def __init__(self, code, msg):
        super().__init__("libffb6d_b200 error %d: %s" % (code, msg))
        self.code = code


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "%s not found: the CUDA library has not been built (run __graft_entry__.build() "
            "or `make -C ffb6d_b200/csrc`). There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp, i64, sz, ci, fp, dp = C.c_void_p, C.c_int64, C.c_size_t, C.c_int, C.c_float, C.c_double
    sig = {
        "ffb6d_version": (ci, []),
        "ffb6d_last_error": (C.c_char_p, []),
        "ffb6d_device_count": (ci, []),
        "ffb6d_launch_count": (C.c_uint64, []),
        "ffb6d_knn_workspace_bytes": (sz, [i64, i64, i64, ci]),
        "ffb6d_knn_batch": (ci, [vp, vp, i64, i64, i64, ci, vp, ci, vp, sz, vp]),
        "ffb6d_knn_batch_algo": (ci, [vp, vp, i64, i64, i64, ci, vp, ci, vp, sz, ci, vp]),
        "ffb6d_knn_grid_bytes": (sz, [i64, i64]),
        "ffb6d_knn_grid_query_bytes": (sz, [i64, i64]),
        "ffb6d_knn_grid_build": (ci, [vp, i64, i64, ci, vp, sz, vp]),
        "ffb6d_knn_grid_query": (ci, [vp, vp, i64, i64, i64, ci, vp, ci, vp, sz, vp, sz, vp]),
        "ffb6d_knn_grid_query_organized": (ci, [vp, vp, i64, i64, i64, ci, vp, ci, vp, sz, vp, sz, i64, vp]),
        "ffb6d_knn_subset_nn": (ci, [vp, vp, i64, i64, i64, vp, ci, vp, ci, vp, sz, vp]),
        "ffb6d_build_indices_workspace_bytes": (sz, [i64, i64, i64, i64, ci]),
        "ffb6d_build_indices": (ci, [vp, vp, vp, vp, i64, i64, i64, i64, ci, vp, ci, vp, sz, vp]),
        "ffb6d_knn_grid_tune": (None, [fp, ci]),
        "ffb6d_knn_grid_tune_k1": (None, [fp]),
        "ffb6d_knn_batch_host": (ci, [vp, sz, sz, sz, vp, sz, sz, vp]),
        "ffb6d_knn_host": (ci, [vp, sz, sz, vp, sz, sz, vp]),
        "ffb6d_gather_max_fwd": (ci, [vp, vp, ci, i64, i64, i64, i64, ci, ci, vp, vp]),
        "ffb6d_check_indices": (ci, [vp, ci, i64, i64, vp]),
        "ffb6d_gather_kernel_name": (C.c_char_p, [i64, i64, i64, i64, ci, ci]),
        "ffb6d_gather_max_bwd": (ci, [vp, vp, ci, vp, i64, i64, i64, i64, ci, ci, vp, vp]),
        "ffb6d_gather_neighbour_fwd": (ci, [vp, vp, ci, i64, i64, i64, i64, ci, vp, vp]),
        "ffb6d_gather_neighbour_bwd": (ci, [vp, vp, ci, i64, i64, i64, i64, ci, vp, vp]),
        "ffb6d_relative_pos_encoding_fwd": (ci, [vp, vp, ci, i64, i64, ci, vp, vp]),
        "ffb6d_fusion_mlp_fwd": (ci, [vp, i64, vp, i64, vp, vp, vp, i64, i64, i64, ci, fp, vp, vp]),
        "ffb6d_fusion_mlp_pack_bytes": (sz, [i64, i64]),
        "ffb6d_fusion_mlp_pack": (ci, [vp, i64, i64, vp, sz, vp]),
        "ffb6d_fusion_mlp_fwd_packed": (ci, [vp, i64, vp, i64, vp, vp, vp, i64, i64, i64, ci, fp, vp, vp]),
        "ffb6d_fusion_mlp_fwd_ex": (ci, [vp, i64, vp, i64, vp, vp, vp, i64, i64, i64, ci, fp, vp, vp, ci, i64, ci, vp, vp]),
        "ffb6d_bn_workspace_bytes": (sz, [i64, i64]),
        "ffb6d_bn_train_fwd": (ci, [vp, i64, i64, i64, vp, vp, fp, fp, vp, vp, ci, fp, vp, vp, vp, sz, vp]),
        "ffb6d_bn_train_bwd": (ci, [vp, vp, vp, i64, i64, i64, ci, fp, vp, vp, vp, vp, sz, vp]),
        "ffb6d_bn_train_stats": (ci, [vp, i64, i64, i64, vp, vp, sz, vp]),
        "ffb6d_bn_train_apply": (ci, [vp, i64, i64, i64, vp, dp, vp, vp, fp, fp, vp, vp, ci, fp, vp, vp, vp]),
        "ffb6d_bn_train_bwd_stats": (ci, [vp, vp, vp, i64, i64, i64, ci, fp, vp, vp, vp, vp, sz, vp]),
        "ffb6d_bn_train_bwd_apply": (ci, [vp, vp, vp, vp, dp, i64, i64, i64, ci, fp, vp, vp]),
        "ffb6d_act_bwd": (ci, [vp, vp, i64, ci, fp, vp, vp]),
        "ffb6d_fusion_mlp_wgrad": (ci, [vp, vp, i64, vp, i64, i64, i64, i64, vp, vp]),
        "ffb6d_att_pool_bwd": (ci, [vp, i64, vp, i64, vp, vp, i64, i64, ci, vp, vp, vp, vp]),
        "ffb6d_lfa_att_pool_fused": (ci, [vp, vp, ci, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, i64, ci, i64, i64, fp, vp, vp]),
        "ffb6d_att_pool_fwd": (ci, [vp, i64, vp, i64, vp, i64, i64, ci, vp, vp]),
        "ffb6d_relative_pos_encoding_cm_fwd": (ci, [vp, vp, ci, i64, i64, ci, vp, vp]),
        "ffb6d_backproject": (ci, [vp, i64, i64, i64, vp, ci, vp, i64, vp, vp, vp, vp, vp]),
        "ffb6d_sample_pixels_workspace_bytes": (sz, [i64, i64, i64]),
        "ffb6d_sample_pixels": (ci, [vp, i64, i64, i64, fp, i64, C.c_uint64, vp, vp, vp, sz, vp]),
        "ffb6d_mean_shift_workspace_bytes": (sz, [i64, i64]),
        "ffb6d_mean_shift_fit": (ci, [vp, vp, i64, i64, i64, fp, ci, vp, vp, vp, vp, vp, sz, vp]),
        "ffb6d_best_fit_transform": (ci, [vp, vp, i64, i64, vp, vp]),
        "ffb6d_grid_subsample_host": (ci, [vp, sz, vp, sz, vp, sz, fp, vp, vp, vp, C.POINTER(sz)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    return lib, sorted(sig)


lib, SYMBOLS = _load()


def last_error():
    return lib.ffb6d_last_error().decode("utf-8", "replace")


def check(rc):
    if rc != OK:
        raise FFB6DError(rc, last_error())


def launch_count():
    return int(lib.ffb6d_launch_count())
