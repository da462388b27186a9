"""ctypes binding of libmalstroem_b200.so (include/malstroem_b200.h).

There is no CPU fallback: if the shared library is missing, or no CUDA device is present when a
function is called, the call raises.
"""
import ctypes
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MS_LIB") or os.path.join(_HERE, "libmalstroem_b200.so")

MS_F32, MS_F64, MS_U8, MS_I32, MS_I64 = 0, 1, 2, 3, 4
DTYPE_CODE = {np.dtype(np.float32): MS_F32, np.dtype(np.float64): MS_F64, np.dtype(np.uint8): MS_U8,
              np.dtype(np.bool_): MS_U8, np.dtype(np.int32): MS_I32, np.dtype(np.int64): MS_I64}

ERR_CUDA, ERR_ARG, ERR_SHAPE, ERR_LABEL, ERR_NOCONV = -1, -2, -3, -4, -5
MS_FLOOD_LABEL, MS_FLOOD_UNIFORM, MS_FLOOD_VOLUME, MS_FLOOD_SIZE, MS_FLOOD_CAPACITY = 1, 2, 4, 8, 16   # ms_band_flood_*_dev

c_i64 = ctypes.c_int64
c_int = ctypes.c_int
c_dbl = ctypes.c_double
c_p = ctypes.c_void_p

# every exported symbol of include/malstroem_b200.h: (restype, argtypes)
SIGNATURES = {
    "ms_version": (c_int, []),
    "ms_init": (c_int, [c_int]),
    "ms_shutdown": (c_int, []),
    "ms_cache_clear": (c_int, []),
    "ms_cache_forget": (c_int, [c_p]),
    "ms_cache_stats": (c_int, [c_p]),
    "ms_last_error": (ctypes.c_char_p, []),
    "ms_device_count": (c_int, []),
    "ms_kernel_launches": (c_i64, [c_int]),
    "ms_profile": (c_int, [c_int]),
    "ms_host_counters": (c_int, [c_p, c_int]),
    "ms_profile_report": (c_int, [ctypes.c_char_p, c_i64]),
    "ms_host_alloc": (c_p, [c_i64]),
    "ms_host_free": (c_int, [c_p]),
    "ms_fill_terrain": (c_int, [c_p, c_p, c_p, c_i64, c_i64]),
    "ms_fill_terrain_dev": (c_int, [c_p, c_p, c_p, c_i64, c_i64, c_p]),
    "ms_minmax_f32": (c_int, [c_p, c_i64, c_p, c_p]),
    "ms_minmax_f32_dev": (c_int, [c_p, c_i64, c_p, c_p]),
    "ms_fill_terrain_no_flats": (c_int, [c_p, c_dbl, c_dbl, c_p, c_i64, c_i64]),
    "ms_fill_terrain_no_flats_dev": (c_int, [c_p, c_p, c_dbl, c_dbl, c_p, c_i64, c_i64, c_p, c_p]),
    "ms_flowdir": (c_int, [c_p, c_p, c_i64, c_i64, c_int]),
    "ms_flowdir_dev": (c_int, [c_p, c_p, c_i64, c_i64, c_int, c_p]),
    "ms_accumulated_flow": (c_int, [c_p, c_p, c_i64, c_i64]),
    "ms_accumulated_flow_dev": (c_int, [c_p, c_p, c_i64, c_i64, c_p]),
    "ms_watersheds_from_labels": (c_int, [c_p, c_p, c_int, c_i64, c_i64, c_i64]),
    "ms_watersheds_from_labels_dev": (c_int, [c_p, c_p, c_int, c_i64, c_i64, c_i64, c_p]),
    "ms_connected_components": (c_int, [c_p, c_int, c_p, c_i64, c_i64, c_p]),
    "ms_connected_components_dev": (c_int, [c_p, c_int, c_p, c_i64, c_i64, c_p, c_p]),
    "ms_label_range": (c_int, [c_p, c_i64, c_p, c_p]),
    "ms_label_range_dev": (c_int, [c_p, c_i64, c_p, c_p]),
    "ms_label_stats": (c_int, [c_p, c_int, c_p, c_i64, c_i64, c_p, c_p, c_p, c_p]),
    "ms_label_stats_dev": (c_int, [c_p, c_int, c_p, c_i64, c_i64, c_p, c_p, c_p, c_p, c_p]),
    "ms_label_extreme_index": (c_int, [c_p, c_p, c_i64, c_i64, c_i64, c_int, c_p, c_p, c_p]),
    "ms_label_extreme_index_dev": (c_int, [c_p, c_p, c_i64, c_i64, c_i64, c_int, c_p, c_p, c_p, c_p]),
    "ms_label_count": (c_int, [c_p, c_i64, c_i64, c_p]),
    "ms_label_count_dev": (c_int, [c_p, c_i64, c_i64, c_p, c_p]),
    "ms_keep_labels": (c_int, [c_p, c_i64, c_p, c_i64, c_p]),
    "ms_keep_labels_dev": (c_int, [c_p, c_i64, c_p, c_i64, c_p, c_p]),
    "ms_band_create": (c_int, [c_i64, c_i64, c_int, c_p]),
    "ms_band_destroy": (c_int, [c_p]),
    "ms_band_fill_local_dev": (c_int, [c_p, c_p, c_p, c_p]),
    "ms_band_fill_edge_ids_dev": (c_int, [c_p, c_i64, c_p, c_p, c_p]),
    "ms_band_fill_edges_dev": (c_int, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i64, c_p, c_p]),
    "ms_graph_minimax_dev": (c_int, [c_i64, c_p, c_p, c_p, c_i64, c_p, c_p]),
    "ms_band_fill_finish_dev": (c_int, [c_p, c_p, c_p, c_p, c_p, c_p]),
    "ms_nf_cap_bound": (c_dbl, [c_i64, c_i64, c_dbl]),
    "ms_band_nf_init_dev": (c_int, [c_p, c_p, c_p, c_p, c_p, c_p]),
    "ms_band_nf_solve_dev": (c_int, [c_p, c_p, c_p, c_p, c_dbl, c_dbl, c_dbl, c_int, c_int, c_int, c_p, c_p]),
    "ms_band_nf_verify_dev": (c_int, [c_p, c_p, c_p, c_dbl, c_dbl, c_p, c_p]),
    "ms_band_nf_ban_dev": (c_int, [c_p, c_p, c_p, c_dbl, c_dbl, c_int, c_p, c_p]),
    "ms_band_nf_shared_create": (c_int, [c_p, c_p]),
    "ms_band_nf_shared_open": (c_int, [c_p, c_int, c_int, c_p, c_p]),
    "ms_band_nf_p2p_arm_dev": (c_int, [c_p, c_p]),
    "ms_band_nf_ir_edgefix_dev": (c_int, [c_p, c_p, c_p, c_p, c_p, c_p]),
    "ms_band_nf_ir_prepare_dev": (c_int, [c_p, c_p, c_p, c_dbl, c_dbl, c_dbl, c_p, c_p, c_p, c_p, c_p]),
    "ms_band_nf_ir_solve_launch_dev": (c_int, [c_p, c_p, c_dbl, c_dbl, c_p]),
    "ms_band_nf_ir_solve_wait_dev": (c_int, [c_p, c_p, c_p, c_p]),
    "ms_band_nf_ir_finish_dev": (c_int, [c_p, c_p, c_p, c_p, c_p, c_dbl, c_dbl, c_p, c_p]),
    "ms_band_flowdir_dev": (c_int, [c_p, c_p, c_p, c_int, c_p]),
    "ms_band_accum_local_dev": (c_int, [c_p, c_p, c_p, c_p, c_p, c_p]),
    "ms_forest_accumulate_dev": (c_int, [c_i64, c_p, c_p, c_p]),
    "ms_band_accum_finish_dev": (c_int, [c_p, c_p, c_p, c_p, c_p, c_p]),
    "ms_band_cc_local_dev": (c_int, [c_p, c_p, c_int, c_i64, c_p, c_p, c_p]),
    "ms_cc_boundary_merge": (c_int, [c_int, c_i64, c_p, c_p, c_p, c_p, c_i64, c_p]),
    "ms_cc_boundary_merge_values": (c_int, [c_int, c_i64, c_p, c_p, c_p, c_p, c_int, c_p, c_p, c_i64, c_p]),
    "ms_band_cc_count_dev": (c_int, [c_p, c_p, c_i64, c_p, c_p]),
    "ms_band_cc_root_labels_dev": (c_int, [c_p, c_p, c_i64, c_i64, c_p, c_p]),
    "ms_band_cc_finish_dev": (c_int, [c_p, c_p, c_p, c_i64, c_i64, c_p, c_p]),
    "ms_band_ws_local_dev": (c_int, [c_p, c_p, c_p, ctypes.c_int32, c_p, c_p, c_p]),
    "ms_chain_resolve_dev": (c_int, [c_i64, c_p, c_p, c_p]),
    "ms_band_ws_finish_dev": (c_int, [c_p, c_p, c_p, ctypes.c_int32, c_p, c_p]),
    "ms_band_tables_a_dev": (c_int, [c_p, c_p, c_p, c_p, c_p, c_i64, c_i64, c_i64, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
    "ms_band_tables_b_dev": (c_int, [c_p, c_p, c_p, c_i64, c_i64, c_p, c_p, c_i64, c_p, c_p, c_p]),
    "ms_pipeline_dev": (c_int, [c_p, c_p]),
    "ms_pipeline_host_dev": (c_int, [c_p, c_p, c_p]),
    "ms_pipeline_filtered_host_dev": (c_int, [c_p, c_p, c_p, c_p, c_p]),
    "ms_bluespot_filter_dev": (c_int, [c_p, c_i64, c_p, c_p, c_p, c_p, c_p, c_p]),
    "ms_relabel_dev": (c_int, [c_p, c_i64, c_i64, c_p, c_p]),
    "ms_copies_wait": (c_int, []),
    "ms_synth_fractal_dev": (c_int, [c_p, c_i64, c_i64, c_i64, c_i64, c_int, c_p]),
    "ms_pourpoint_network": (c_int, [c_p, c_p, c_int, c_i64, c_i64, c_i64, c_p, c_p, c_i64, c_int, c_p, c_p, c_p, c_p,
                                     c_i64]),
    "ms_pourpoint_network_dev": (c_int, [c_p, c_p, c_int, c_i64, c_i64, c_i64, c_p, c_p, c_i64, c_int, c_p, c_p, c_p]),
    "ms_rain_events": (c_int, [c_i64, c_p, c_p, c_p, c_i64, c_p, c_int, c_p, c_p, c_p, c_p, c_p]),
    "ms_rain_events_dev": (c_int, [c_i64, c_p, c_p, c_p, c_i64, c_p, c_int, c_p, c_p, c_p, c_p, c_p, c_p]),
    "ms_band_pp_parent_dev": (c_int, [c_p, c_p, c_p, c_p, c_i64, c_i64, c_i64, c_i64, c_i64, c_p, c_p, c_p, c_p]),
    "ms_tiff_tile_slot": (c_i64, [c_int]),
    "ms_tiff_encode_dev": (c_int, [c_p, c_int, c_i64, c_i64, c_int, c_p, c_i64, c_p, c_p]),
    "ms_tiff_pack_dev": (c_int, [c_p, c_i64, c_p, c_p, c_i64, c_p, c_p]),
    "ms_tiff_decode_dev": (c_int, [c_p, c_p, c_p, c_i64, c_int, c_int, c_int, c_int, c_int, c_p, c_p, c_i64, c_i64,
                                   c_int, c_dbl, c_dbl, c_int, c_p]),
    "ms_tiff_decode_rows_dev": (c_int, [c_p, c_p, c_p, c_i64, c_int, c_int, c_int, c_int, c_int, c_p, c_p, c_i64,
                                        c_i64, c_i64, c_i64, c_i64, c_int, c_dbl, c_dbl, c_int, c_p]),
    "ms_polygonize_dev": (c_int, [c_p, c_i64, c_i64, c_int, c_int, ctypes.c_int32, c_p, c_p]),
    "ms_polygonize": (c_int, [c_p, c_i64, c_i64, c_int, c_int, ctypes.c_int32, c_p]),
    "ms_polygonize_fetch": (c_int, [c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
    "ms_band_poly_count_dev": (c_int, [c_p, c_i64, c_i64, c_int, c_int, c_int, ctypes.c_int32, c_p, c_p, c_p, c_p, c_p]),
    "ms_band_poly_edges_dev": (c_int, [c_p, c_i64, c_i64, c_int, c_int, c_int, ctypes.c_int32, c_p, c_i64, c_p, c_p, c_p,
                                       c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
    "ms_band_poly_place_dev": (c_int, [c_i64, c_i64, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p,
                                       c_p, c_p]),
    "ms_band_poly_emit_dev": (c_int, [c_p, c_i64, c_i64, c_int, c_int, c_int, ctypes.c_int32, c_i64, c_i64, c_p, c_p, c_p,
                                      c_p, c_p, c_p, c_p, c_p, c_p, c_i64, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p,
                                      c_p, c_p]),
    "ms_bluespot_network_dev": (c_int, [c_p, c_dbl, c_int, c_i64, c_p, c_int, c_p, c_p, c_p, c_p, c_p, c_p]),
    "ms_flood_levels_dev": (c_int, [c_p, c_p, c_p, c_i64, c_i64, c_i64, c_p, c_dbl, c_i64, c_p, c_p, c_p, c_p]),
    "ms_flood_levels": (c_int, [c_p, c_p, c_p, c_i64, c_i64, c_i64, c_p, c_dbl, c_i64, c_p, c_p, c_p]),
    "ms_water_depth_dev": (c_int, [c_p, c_p, c_p, c_i64, c_i64, c_i64, c_p, c_p, c_p]),
    "ms_water_depth": (c_int, [c_p, c_p, c_p, c_i64, c_i64, c_i64, c_p, c_p]),
    "ms_band_flood_count_dev": (c_int, [c_p, c_p, c_p, c_i64, c_i64, c_i64, c_i64, c_i64, c_p, c_p, c_p, c_p, c_i64,
                                        c_p, c_p, c_p, c_p]),
    "ms_band_flood_layout_dev": (c_int, [c_i64, c_i64, c_i64, c_p, c_p, c_p, c_p, c_i64, c_p, c_p, c_p, c_p]),
    "ms_band_flood_scatter_dev": (c_int, [c_p, c_p, c_p, c_i64, c_i64, c_i64, c_i64, c_i64, c_p, c_p, c_p, c_p, c_p,
                                          c_p, c_p]),
    "ms_band_flood_solve_dev": (c_int, [c_i64, c_i64, c_i64, c_p, c_p, c_p, c_p, c_i64, c_p, c_p, c_i64, c_p, c_dbl,
                                        c_i64, c_p, c_p, c_p, c_p, c_p]),
}


class MsRasters(ctypes.Structure):
    """struct ms_rasters of include/malstroem_b200.h"""
    _fields_ = [("rows", c_i64), ("cols", c_i64),
                ("dem", c_p), ("filled", c_p), ("depths", c_p), ("fnf", c_p), ("flowdir", c_p), ("accum", c_p),
                ("labels", c_p), ("wsheds", c_p),
                ("table_capacity", c_i64),
                ("st_min", c_p), ("st_max", c_p), ("st_sum", c_p), ("st_count", c_p), ("ws_count", c_p),
                ("ppmin_value", c_p), ("ppmin_row", c_p), ("ppmin_col", c_p),
                ("ppmax_value", c_p), ("ppmax_row", c_p), ("ppmax_col", c_p),
                ("nlabels", c_i64), ("short_eps", c_dbl), ("diag_eps", c_dbl), ("stats", c_i64 * 8)]


class MsHostOut(ctypes.Structure):
    """struct ms_host_out of include/malstroem_b200.h"""
    _fields_ = [("filled", c_p), ("depths", c_p), ("fnf", c_p), ("flowdir", c_p), ("accum", c_p), ("labels", c_p),
                ("wsheds", c_p)]


MS_BF_MAX_OPS, MS_BF_MAX_STACK = 64, 16


class MsBluespotFilter(ctypes.Structure):
    """struct ms_bluespot_filter of include/malstroem_b200.h (malstroem_b200.bluespot_filter builds it)"""
    _fields_ = [("n_ops", ctypes.c_int32), ("op", ctypes.c_int32 * MS_BF_MAX_OPS), ("imm", c_dbl * MS_BF_MAX_OPS),
                ("cell_area", c_dbl)]


_lib = None
lock = threading.RLock()      # ctypes drops the GIL; the library keeps per-process state


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("malstroem_b200: %s is missing — build it with `python malstroem_b200/build.py` "
                              "(there is no CPU fallback)" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def check(rc, what=""):
    if rc == 0:
        return
    msg = lib().ms_last_error().decode("utf-8", "replace")
    if rc in (ERR_ARG, ERR_SHAPE):
        raise ValueError("%s: %s" % (what, msg))
    if rc == ERR_LABEL:
        raise IndexError("%s: %s" % (what, msg))
    raise RuntimeError("%s: %s (code %d)" % (what, msg, rc))


def ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


# ---- device twins of host rasters (csrc/cache.cu) ------------------------------------------------------------------
# The library keys a twin on the host address; numpy hands a freed array's address out again, so every array that
# went through a host-pointer call gets a finalizer that tells the library when the array object dies.
import weakref  # noqa: E402

_tracked = {}


def _forget(address, key):
    _tracked.pop(key, None)
    if _lib is not None:
        with lock:
            _lib.ms_cache_forget(ctypes.c_void_p(address))


def track(*arrays):
    """Call after a host-pointer entry point with the raster arrays it read or wrote."""
    for a in arrays:
        if not isinstance(a, np.ndarray) or a.size < 4096:
            continue
        key = id(a)
        if key in _tracked:
            continue
        try:
            _tracked[key] = weakref.finalize(a, _forget, a.ctypes.data, key)
        except TypeError:
            pass


# ---- result arrays in pinned host memory ------------------------------------------------------------------------------
# A device-to-host copy into a freshly allocated pageable numpy array runs at ~4.5 GB/s on the B200 boxes (page faults
# + the driver's staging copies); into pinned memory at ~50 GB/s.  The result arrays of the mirrors are ours to
# allocate, so they come from a pool of pinned buffers (ms_host_alloc) that take a buffer back when the array (and every
# view of it) has died - the second fill_terrain_no_flats of a run lands in the buffer the first one used.
# MS_PINNED_GB (default 24) caps the pool; beyond it, or with MS_PINNED=0, results are plain numpy arrays.
_pin_pool = {}           # nbytes -> [address]
_pin_total = [0]
_PIN_MIN = 1 << 20


def _pin_release(address, nbytes):
    _pin_pool.setdefault(nbytes, []).append(address)


def result_array(shape, dtype):
    """np.empty(shape, dtype) in pinned host memory where possible (see above)."""
    dtype = np.dtype(dtype)
    nbytes = int(np.prod(shape)) * dtype.itemsize
    if nbytes < _PIN_MIN or os.environ.get("MS_PINNED", "1") == "0" or _lib is None:
        return np.empty(shape, dtype)
    free = _pin_pool.get(nbytes)
    if free:
        address = free.pop()
    else:
        cap = float(os.environ.get("MS_PINNED_GB", "24")) * 1e9
        if _pin_total[0] + nbytes > cap:
            # give back what the pool holds in other sizes before giving up on pinned memory
            for size, lst in list(_pin_pool.items()):
                while lst:
                    _lib.ms_host_free(ctypes.c_void_p(lst.pop()))
                    _pin_total[0] -= size
            if _pin_total[0] + nbytes > cap:
                return np.empty(shape, dtype)
        with lock:
            address = _lib.ms_host_alloc(nbytes)
        if not address:
            return np.empty(shape, dtype)
        _pin_total[0] += nbytes
    buf = (ctypes.c_char * nbytes).from_address(address)
    weakref.finalize(buf, _pin_release, address, nbytes)        # fires when the last array over the buffer is gone
    return np.frombuffer(buf, dtype=dtype).reshape(shape)


def cache_clear():
    """Forget every device twin (call after rewriting an array in place between two plug-in calls)."""
    with lock:
        check(lib().ms_cache_clear(), "ms_cache_clear")


def cache_stats():
    out = (ctypes.c_int64 * 5)()
    with lock:
        check(lib().ms_cache_stats(out), "ms_cache_stats")
    return dict(zip(("input_hits", "input_uploads", "derived_hits", "evictions", "bytes"), [int(v) for v in out]))
