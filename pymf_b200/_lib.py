"""ctypes binding of libpymfb.so (C ABI in include/pymfb.h).

The library is built in-tree by ``pymf_b200/csrc/build.sh`` (see ``__graft_entry__.build``).
There is no CPU fallback: if the shared object is missing, or no B200 is visible, the
product raises instead of computing anything on the host.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PYMFB_LIB: alternative build of the same library (kernel experiments: ablation variants built with
# PYMFB_NVCC_EXTRA / PYMFB_OUT); the default is the in-tree product library.
LIB_PATH = os.environ.get("PYMFB_LIB") or os.path.join(_HERE, "libpymfb.so")

F32, F64 = 0, 1
I32, I64 = 2, 3
LAYOUT_COO, LAYOUT_CSR, LAYOUT_CSC = 0, 1, 2
COMPUTE_W, COMPUTE_H, COMPUTE_ERR, EARLY_STOP = 1, 2, 4, 8
PATH_AUTO, PATH_SIMT, PATH_TC, PATH_SPARSE = 0, 1, 2, 3
OPT_PATH = 1
OPT_ERR_MODE = 2
OPT_GRAPH = 3
OPT_NNDSVD_PATH = 4
GRAPH_AUTO, GRAPH_OFF, GRAPH_ON = 0, 1, 2
VARIANT_NMF, VARIANT_SNMF = 0, 1
ERR_AUTO, ERR_TRACE, ERR_DIRECT = 0, 1, 2

_c_ctx = C.c_void_p
_i64 = C.c_int64

# name -> (restype, argtypes); must list every symbol include/pymfb.h declares
SIGNATURES = {
    "pymfb_version": (C.c_int, []),
    "pymfb_last_error": (C.c_char_p, []),
    "pymfb_device_count": (C.c_int, []),
    "pymfb_create": (C.c_int, [C.POINTER(_c_ctx), C.c_int, _i64, _i64, _i64, _i64, C.c_int]),
    "pymfb_destroy": (C.c_int, [_c_ctx]),
    "pymfb_set_option": (C.c_int, [_c_ctx, C.c_int, _i64]),
    "pymfb_set_penalty": (C.c_int, [_c_ctx, C.c_double, C.c_double, C.c_double, C.c_double]),
    "pymfb_set_variant": (C.c_int, [_c_ctx, C.c_int]),
    "pymfb_get_penalty": (C.c_int, [_c_ctx, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "pymfb_comm_unique_id": (C.c_int, [C.c_void_p]),
    "pymfb_comm_init": (C.c_int, [_c_ctx, C.c_void_p, C.c_int, C.c_int]),
    "pymfb_comm_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_int, C.c_int]),
    "pymfb_comm_attach": (C.c_int, [_c_ctx, C.c_void_p, C.c_int, C.c_int]),
    "pymfb_comm_destroy": (C.c_int, [C.c_void_p]),
    "pymfb_bind_x": (C.c_int, [_c_ctx, C.c_void_p, _i64]),
    "pymfb_upload_x": (C.c_int, [_c_ctx, C.c_void_p, C.c_int, _i64]),
    "pymfb_gen_x": (C.c_int, [_c_ctx, C.c_uint64]),
    "pymfb_upload_x_csc": (C.c_int, [_c_ctx, C.POINTER(_i64), C.POINTER(C.c_int32), C.c_void_p, C.c_int, _i64]),
    "pymfb_upload_x_sparse_device": (C.c_int, [_c_ctx, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                               C.c_int, _i64]),
    "pymfb_host_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_size_t]),
    "pymfb_host_free": (C.c_int, [C.c_void_p]),
    "pymfb_last_upload_pinned": (C.c_int, [_c_ctx]),
    "pymfb_upload_x_begin": (C.c_int, [_c_ctx]),
    "pymfb_upload_x_panel": (C.c_int, [_c_ctx, C.c_void_p, C.c_int, _i64, _i64, _i64, C.c_int]),
    "pymfb_upload_x_wait": (C.c_int, [_c_ctx, C.c_int]),
    "pymfb_upload_x_end": (C.c_int, [_c_ctx]),
    "pymfb_device_numa_node": (C.c_int, [C.c_int]),
    "pymfb_host_node_of": (C.c_int, [C.c_void_p]),
    "pymfb_set_w": (C.c_int, [_c_ctx, C.c_void_p, C.c_int]),
    "pymfb_set_h": (C.c_int, [_c_ctx, C.c_void_p, C.c_int]),
    "pymfb_get_w": (C.c_int, [_c_ctx, C.c_void_p, C.c_int]),
    "pymfb_get_h": (C.c_int, [_c_ctx, C.c_void_p, C.c_int]),
    "pymfb_gen_w": (C.c_int, [_c_ctx, C.c_uint64]),
    "pymfb_gen_h": (C.c_int, [_c_ctx, C.c_uint64]),
    "pymfb_run": (C.c_int, [_c_ctx, C.c_int, C.c_uint, C.POINTER(C.c_double),
                            C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "pymfb_frobenius": (C.c_int, [_c_ctx, C.POINTER(C.c_double)]),
    "pymfb_nndsvd": (C.c_int, [_c_ctx, C.c_int, C.c_double, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_double)]),
    "pymfb_nndsvd_info": (C.c_int, [_c_ctx, C.POINTER(C.c_int), C.POINTER(C.c_double)]),
    "pymfb_enqueue": (C.c_int, [_c_ctx, C.c_int, C.c_uint]),
    "pymfb_sync": (C.c_int, [_c_ctx]),
    "pymfb_stream": (C.c_void_p, [_c_ctx]),
    "pymfb_event_create": (C.c_int, [C.POINTER(C.c_void_p)]),
    "pymfb_event_record": (C.c_int, [_c_ctx, C.c_void_p]),
    "pymfb_event_elapsed_ms": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_float)]),
    "pymfb_event_destroy": (C.c_int, [C.c_void_p]),
    "pymfb_kernel_timing": (C.c_int, [_c_ctx, C.c_int]),
    "pymfb_kernel_timing_read": (C.c_int, [_c_ctx, C.c_int, C.POINTER(C.c_double), C.POINTER(_i64)]),
    "pymfb_launch_count": (_i64, [_c_ctx]),
    "pymfb_graph_replays": (_i64, [_c_ctx]),
    "pymfb_active_path": (C.c_int, [_c_ctx]),
    "pymfb_flush_l2": (C.c_int, [_c_ctx]),
}

_lib = None


class PymfbError(RuntimeError):
    pass


def load():
    """Load libpymfb.so (once) and declare all signatures.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise PymfbError(
            "libpymfb.so is not built (%s missing): run `python -c 'import __graft_entry__ as g; "
            "g.build()'` or pymf_b200/csrc/build.sh.  There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().pymfb_last_error()
        raise PymfbError(msg.decode("utf-8", "replace") if msg else "libpymfb call failed (%d)" % rc)


def device_count():
    return int(load().pymfb_device_count())
