"""ctypes binding of librange_b200.so (C ABI: include/range_b200.h).

There is NO fallback: if the CUDA extension is missing or a call fails this module raises.
"""
import ctypes
import os
from ctypes import (POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_void_p)

_HERE = os.path.dirname(os.path.abspath(__file__))
# RANGE_B200_LIB: developer switch (tools/variants.sh builds the library with other tuning macros for A/B timing)
LIB_PATH = os.environ.get("RANGE_B200_LIB") or os.path.join(_HERE, "librange_b200.so")

RANGE_MODE_RANGE, RANGE_MODE_RANGE_PLUS = 0, 1
RANGE_OUT_F64, RANGE_OUT_F32, RANGE_OUT_PACKED = 0, 1, 2
RANGE_MAX_RANKS = 8
RANGE_ENC_F64, RANGE_ENC_F16X3 = 0, 1
RANGE_TOPK_MAX = 32
RANGE_SWEEP_MAX_BETAS = 8

# every symbol include/range_b200.h declares: name -> (restype, argtypes)
PROTOTYPES = {
    "range_last_error": (c_char_p, []),
    "range_version": (c_int, []),
    "range_launch_count": (c_int64, []),
    "range_ctx_create": (c_int, [c_int, POINTER(c_void_p)]),
    "range_ctx_destroy": (c_int, [c_void_p]),
    "range_ctx_set_sh_table": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "range_ctx_set_sh_closed_form": (c_int, [c_void_p, c_int, c_int, c_void_p]),
    "range_ctx_set_encoder": (c_int, [c_void_p, c_int, POINTER(c_int32), POINTER(c_void_p), POINTER(c_void_p),
                                      c_double, c_double]),
    "range_encoder_prepared_bytes": (c_size_t, [c_void_p]),
    "range_ctx_prepare_encoder": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
    "range_ctx_set_encoder_precision": (c_int, [c_void_p, c_int]),
    "range_ctx_set_db": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_float]),
    "range_ctx_set_db_caps": (c_int, [c_void_p, c_int64, c_void_p, c_int64]),
    "range_geo_mask_shape": (c_int, [c_void_p, c_int64, POINTER(c_int32), POINTER(c_int32)]),
    "range_geo_mask": (c_int, [c_void_p, c_int64, c_void_p, c_float, c_void_p, c_void_p, c_void_p]),
    "range_sort_workspace_bytes": (c_size_t, [c_void_p, c_int64]),
    "range_sort_queries": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "range_sh_features": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p]),
    "range_encode_workspace_bytes": (c_size_t, [c_void_p, c_int64]),
    "range_encode": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                             c_void_p]),
    "range_raster_tables_bytes": (c_size_t, [c_void_p, c_int64, c_int64]),
    "range_raster_tables": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_size_t, c_void_p]),
    "range_raster_points": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p,
                                    c_void_p]),
    "range_encode_raster": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_size_t, c_void_p]),
    "range_retrieve_workspace_bytes": (c_size_t, [c_void_p, c_int64]),
    "range_retrieve_stats": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_float, c_float, c_void_p,
                                     c_void_p, c_void_p, c_size_t, c_void_p]),
    "range_retrieve_apply": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_float, c_float, c_float,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "range_retrieve_apply_concat": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_float, c_float, c_float,
                                            c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_size_t,
                                            c_void_p]),
    "range_retrieve": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_float, c_float, c_float, c_void_p,
                               c_void_p, c_size_t, c_void_p]),
    "range_retrieve_concat": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_float, c_float, c_float, c_void_p,
                                      c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "range_topk_workspace_bytes": (c_size_t, [c_void_p, c_int64, c_int]),
    "range_retrieve_topk": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_float, c_float, c_float, c_void_p,
                                    c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "range_retrieve_topk_rows": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_float, c_float, c_float,
                                         c_void_p, c_int, c_int64, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "range_topk_merge": (c_int, [c_void_p, c_int, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_void_p]),
    "range_retrieve_apply_routed": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_float, c_float, c_float,
                                            c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "range_combine_concat": (c_int, [c_void_p, c_int64, c_int, POINTER(c_void_p), POINTER(c_float), c_void_p, c_void_p,
                                     c_void_p, c_int, c_void_p]),
    "range_sweep_concat": (c_int, [c_void_p, c_int64, c_int, POINTER(c_void_p), POINTER(c_void_p), c_int, POINTER(c_float),
                                   POINTER(c_float), c_void_p, c_void_p, POINTER(c_void_p), c_int, c_void_p]),
    "range_peer_alloc": (c_int, [c_size_t, POINTER(c_void_p), c_void_p]),
    "range_peer_open": (c_int, [c_void_p, POINTER(c_void_p)]),
    "range_peer_close": (c_int, [c_void_p]),
    "range_peer_free": (c_int, [c_void_p]),
    "range_host_unpack": (c_int, [c_void_p, c_int64, c_void_p, c_int]),
    "range_concat": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "range_concat_scatter": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
}



class Route(ctypes.Structure):
    """include/range_b200.h: range_route"""
    _fields_ = [("n_ranks", c_int32), ("rank", c_int32), ("slab_rows", c_int64), ("peer", c_void_p * RANGE_MAX_RANKS)]


_lib = None


class RangeError(RuntimeError):
    pass


def load():
    """dlopen the extension (once) and declare every prototype.  Raises if it is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RangeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or range_b200/csrc/build.sh).  range_b200 has no CPU or PyTorch fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def check(code):
    if code != 0:
        raise RangeError(f"librange_b200: error {code}: {load().range_last_error().decode()}")


def launch_count():
    return int(load().range_launch_count())
