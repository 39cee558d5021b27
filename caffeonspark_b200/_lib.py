"""ctypes loader of libcaffedistri_b200.so (built in-tree by csrc/Makefile)."""
import ctypes
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
_LIB = None


def library_path():
    return os.path.join(HERE, "libcaffedistri_b200.so")


def build_library(force=False):
    """nvcc -gencode arch=compute_100a,code=sm_100a build of the shared library."""
    if force:
        subprocess.run(["make", "-s", "-C", CSRC, "clean"], check=True)
    subprocess.run(["make", "-s", "-j8", "-C", CSRC], check=True)
    return library_path()


class cos_blob(ctypes.Structure):
    _fields_ = [("data", ctypes.c_void_p), ("num", ctypes.c_int), ("channels", ctypes.c_int),
                ("height", ctypes.c_int), ("width", ctypes.c_int)]


class cos_solver_desc(ctypes.Structure):
    _fields_ = [("nblobs", ctypes.c_int), ("counts", ctypes.POINTER(ctypes.c_int64)),
                ("lr_mult", ctypes.POINTER(ctypes.c_float)), ("decay_mult", ctypes.POINTER(ctypes.c_float)),
                ("lr_policy", ctypes.c_char_p), ("base_lr", ctypes.c_float), ("gamma", ctypes.c_float),
                ("power", ctypes.c_float), ("stepsize", ctypes.c_int), ("stepvalues", ctypes.POINTER(ctypes.c_int)),
                ("nstepvalues", ctypes.c_int), ("max_iter", ctypes.c_int), ("momentum", ctypes.c_float),
                ("weight_decay", ctypes.c_float), ("test_iter", ctypes.c_int), ("test_interval", ctypes.c_int),
                ("snapshot_prefix", ctypes.c_char_p), ("grad_dtype", ctypes.c_int), ("init_iter", ctypes.c_int),
                ("regularization_l1", ctypes.c_int), ("type", ctypes.c_char_p), ("delta", ctypes.c_float),
                ("rms_decay", ctypes.c_float)]


FORWARD_BACKWARD_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(cos_blob),
                                       ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p)

# every symbol include/caffedistri_b200.h declares: (name, restype, argtypes)
_c = ctypes
_vp, _i, _f, _cp, _i64, _u64 = _c.c_void_p, _c.c_int, _c.c_float, _c.c_char_p, _c.c_int64, _c.c_uint64
_pcp = _c.POINTER(_c.c_char_p)
SYMBOLS = [
    ("cos_last_error", _cp, []),
    ("cos_version", _cp, []),
    ("cos_net_allocate", _i, [_cp, _cp, _cp, _i, _i, _i, _i, _i, _i, _i, _c.POINTER(_vp)]),
    ("cos_net_allocate_desc", _i, [_c.POINTER(cos_solver_desc), _i, _i, _i, _i, _i, _i, _c.POINTER(_vp)]),
    ("cos_net_deallocate", None, [_vp]),
    ("cos_net_local_addresses", _i, [_vp, _c.POINTER(_pcp)]),
    ("cos_net_connect", _i, [_vp, _pcp, _i]),
    ("cos_net_sync", _i, [_vp]),
    ("cos_net_init", _i, [_vp, _i, _i]),
    ("cos_net_train", _i, [_vp, _i, _c.POINTER(cos_blob), _i]),
    ("cos_net_predict", _i, [_vp, _i, _c.POINTER(cos_blob), _i, _pcp, _i, _c.POINTER(cos_blob)]),
    ("cos_net_validation", _i, [_vp, _c.POINTER(cos_blob), _i]),
    ("cos_net_aggregate_validation_outputs", _i, [_vp]),
    ("cos_net_device_id", _i, [_vp, _i]),
    ("cos_net_get_init_iter", _i, [_vp, _i]),
    ("cos_net_get_max_iter", _i, [_vp, _i]),
    ("cos_net_get_test_iter", _i, [_vp, _i]),
    ("cos_net_get_test_interval", _i, [_vp]),
    ("cos_net_snapshot", _i, [_vp]),
    ("cos_net_snapshot_filename", _i, [_vp, _i, _i, _cp, _i]),
    ("cos_caffemodel_write", _i, [_cp, _cp, _i, _pcp, _pcp, _c.POINTER(_i), _c.POINTER(_i64), _c.POINTER(_vp)]),
    ("cos_caffemodel_read", _i64, [_cp, _cp, _i, _vp, _i64]),
    ("cos_solverstate_write", _i, [_cp, _i, _i, _cp, _i, _c.POINTER(_i), _c.POINTER(_i64), _c.POINTER(_vp)]),
    ("cos_solverstate_read", _i64, [_cp, _c.POINTER(_i), _c.POINTER(_i), _cp, _i, _i, _vp, _i64]),
    ("cos_caffemodel_write_h5", _i, [_cp, _i, _pcp, _c.POINTER(_i), _c.POINTER(_i64), _c.POINTER(_vp)]),
    ("cos_solverstate_write_h5", _i, [_cp, _i, _i, _cp, _i, _c.POINTER(_i), _c.POINTER(_i64), _c.POINTER(_vp)]),
    ("cos_hdf5_read_dataset", _i64, [_cp, _cp, _c.POINTER(_i64), _i, _c.POINTER(_i), _vp, _i64]),
    ("cos_net_get_validation_output_blob_names", _i, [_vp, _c.POINTER(_pcp)]),
    ("cos_net_get_validation_output_blobs", _i, [_vp, _i, _c.POINTER(cos_blob)]),
    ("cos_net_set_forward_backward", _i, [_vp, FORWARD_BACKWARD_FN, _vp]),
    ("cos_net_data", _vp, [_vp, _i]),
    ("cos_net_diff", _vp, [_vp, _i]),
    ("cos_net_history", _vp, [_vp, _i]),
    ("cos_net_update_history", _vp, [_vp, _i]),
    ("cos_net_param_count", _i64, [_vp]),
    ("cos_net_shard", _i, [_vp, _i, _c.POINTER(_u64), _c.POINTER(_u64)]),
    ("cos_net_iter", _i, [_vp]),
    ("cos_net_learning_rate", _f, [_vp]),
    ("cos_net_last_loss", _f, [_vp]),
    ("cos_net_sync_step", _i, [_vp, _i, _vp]),
    ("cos_net_all_gather_weights", _i, [_vp, _i, _vp]),
    ("cos_net_synchronize", _i, [_vp]),
    ("cos_net_set_option", _i, [_vp, _cp, _i64]),
    ("cos_net_get_option", _i64, [_vp, _cp]),
    ("cos_net_last_kernel_ms", _f, [_vp]),
    ("cos_net_launch_count", _i64, [_vp]),
    ("cos_net_fill", _i, [_vp, _i, _i, _u64, _u64, _f]),
    ("cos_adapter_create", _vp, [_i, _i]),
    ("cos_adapter_destroy", None, [_vp]),
    ("cos_adapter_address", _cp, [_vp]),
    ("cos_adapter_connect", _i, [_vp, _pcp, _i]),
    ("cos_adapter_barrier", _i, [_vp, _i]),
    ("cos_adapter_offer_fd", _i, [_vp, _cp, _i, _vp, _i]),
    ("cos_adapter_fetch_fd", _i, [_vp, _i, _cp, _vp, _i, _i]),
    ("cos_chunk", None, [_u64, _i, _i, _c.POINTER(_u64), _c.POINTER(_u64)]),
    ("cos_learning_rate", _f, [_cp, _f, _f, _f, _i, _c.POINTER(_i), _i, _i, _i, _c.POINTER(_i)]),
    ("cos_parse_solver", _i, [_cp, _c.POINTER(cos_solver_desc), _c.POINTER(_i64), _c.POINTER(_f), _c.POINTER(_f), _i,
                              _cp, _cp, _i, _c.POINTER(_i), _i, _c.POINTER(_i)]),
]


def lib():
    """Load the CUDA library.  Raises (never falls back) when it is missing."""
    global _LIB
    if _LIB is None:
        path = library_path()
        if not os.path.exists(path):
            raise RuntimeError(
                f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback)")
        L = ctypes.CDLL(path)
        for name, restype, argtypes in SYMBOLS:
            fn = getattr(L, name)  # AttributeError if the ABI lost a symbol
            fn.restype = restype
            fn.argtypes = argtypes
        _LIB = L
    return _LIB
