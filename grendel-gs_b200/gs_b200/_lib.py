"""ctypes binding of the C-ABI library (include/grendel_gs_b200.h).

This is the "reference-side stub" of INTEGRATION.md: plain pointers and sizes go in, torch only
supplies device memory and the current CUDA stream.  There is NO fallback: if the shared library is
missing or a call fails, an exception is raised (the product path never routes through oracle/ or
any CPU implementation).
"""
import ctypes as C
import os

_PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# GS_B200_LIB: a tuning build of the same library (gs_b200.build.build(variant=...)); default = the shipped one
LIB_PATH = os.environ.get("GS_B200_LIB") or os.path.join(_PKG, "lib", "libgrendel_gs_b200.so")

_vp, _i, _f, _i64, _sz = C.c_void_p, C.c_int, C.c_float, C.c_int64, C.c_size_t

# name -> (restype, argtypes); mirrors include/grendel_gs_b200.h declaration by declaration
SIGNATURES = {
    "gs_last_error": (C.c_char_p, []),
    "gs_version": (C.c_char_p, []),
    "gs_get_block_xy": (_i, [C.POINTER(_i)] * 3),
    "gs_preprocess_forward": (_i, [_i, _i, _vp, _vp, _f, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _f,
                                   _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gs_preprocess_backward": (_i, [_i, _i, _vp, _vp, _f, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _f, _vp, _vp,
                                    _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gs_preprocess_forward_raw": (_i, [_i, _i, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _f,
                                       _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gs_preprocess_backward_raw": (_i, [_i, _i, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _f,
                                        _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gs_preprocess_forward_batched": (_i, [_i, _i, _i, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp, _i, _i,
                                           _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gs_preprocess_backward_batched": (_i, [_i, _i, _i, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp, _i, _i, _vp, _vp,
                                            _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gs_get_local2j_ids_bool": (_i, [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "gs_get_local2j_ids_bool_rects": (_i, [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "gs_render_count_temp_bytes": (_sz, [_i]),
    "gs_render_count": (_i, [_i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, C.POINTER(_i64), _vp]),
    "gs_render_sort_temp_bytes": (_sz, [_i64]),
    "gs_render_seg_bytes": (_sz, [_i64, _i]),
    "gs_render_forward": (_i, [_i, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz,
                               _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "gs_render_backward": (_i, [_i, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _vp, _vp, _vp]),
    "gs_render_count_batched": (_i, [_i, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz,
                                     C.POINTER(_i64), _vp]),
    "gs_render_count_launch": (_i, [_i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz,
                                    C.POINTER(C.c_void_p), _vp]),
    "gs_render_count_read": (_i, [_vp, C.POINTER(_i64), _vp]),
    "gs_render_forward_batched": (_i, [_i, _vp, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                       _sz, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "gs_render_backward_batched": (_i, [_i, _i, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _vp,
                                        _vp, _vp]),
    "gs_loss_temp_bytes_batched": (_sz, [_i, _vp, _i]),
    "gs_loss_forward_batched": (_i, [_i, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "gs_loss_backward_batched": (_i, [_i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gs_metrics_batched": (_i, [_i, _i, _i, _vp, _vp, _vp, _i, _vp, _vp]),
    "gs_profile_enable": (_i, [_i]),
    "gs_profile_read": (_i, [_i, C.POINTER(C.c_double), C.POINTER(_i64)]),
    "gs_profile_stage_name": (C.c_char_p, [_i]),
    "gs_debug_set": (_i, [_i]),
    "gs_loss_temp_bytes": (_sz, [_i, _i]),
    "gs_loss_forward": (_i, [_i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "gs_loss_backward": (_i, [_i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gs_route_scan_temp_bytes": (_sz, [_i, _i]),
    "gs_route_scan": (_i, [_i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "gs_xchg_temp_bytes": (_sz, [_i, _i, _i]),
    "gs_xchg_route": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "gs_xchg_pack": (_i, [_i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gs_xchg_unpack": (_i, [_i, _vp, _vp, _vp, _vp, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gs_xchg_pack_grad": (_i, [_i, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "gs_xchg_scatter_grad": (_i, [_i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gs_adam_step": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_float, _vp]),
    "gs_knn3_mean_dist2": (_i, [_i, _vp, _vp, _vp]),
    "gs_densify_temp_bytes": (_sz, [_i]),
    "gs_densify_select": (_i, [_i, _vp, _vp, _vp, _vp, C.c_float, C.c_float, C.c_float, C.c_float, _i, _vp, _sz, _vp, _vp]),
    "gs_densify_gather": (_i, [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gs_peer_alloc": (_i, [_sz, C.POINTER(C.c_void_p), _vp]),
    "gs_peer_open": (_i, [_vp, C.POINTER(C.c_void_p)]),
    "gs_peer_close": (_i, [_vp]),
    "gs_peer_free": (_i, [_vp]),
    "gs_xchg_pack_p2p": (_i, [_i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gs_xchg_pack_grad_p2p": (_i, [_i, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "gs_xr_temp_bytes": (_sz, [_i, _i, _i]),
    "gs_xr_count": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "gs_xr_pack": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_longlong, _vp]),
    "gs_xr_pack_dev": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, C.c_longlong, _vp]),
    "gs_xr_pull_grad": (_i, [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_longlong, _vp, _vp, _vp, _vp]),
    "gs_sparse_grad_mask": (_i, [_i, _vp, _vp, _vp]),
    "gs_sparse_grad_pack": (_i, [_i, _vp, _vp, _vp, _vp, _vp]),
    "gs_sparse_grad_unpack": (_i, [_i, _vp, _vp, _vp, _vp, _vp]),
    "gs_get_touched_locally": (_i, [_i, _i, _i, _vp, _vp, _vp]),
    "gs_get_pixels_compute_locally_and_in_rect": (_i, [_i, _i, _vp, _i, _i, _i, _i, _vp, _vp]),
    "gs_image_tiles_gather": (_i, [_i, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "gs_image_tiles_scatter_add": (_i, [_i, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp]),
}


class GsError(RuntimeError):
    pass


_lib = None


def load():
    """dlopen the in-tree library; raises ImportError (loudly) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU or PyTorch fallback for this operator.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library drift apart
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def call(name, *args):
    """Invoke an int-returning entry point and raise GsError with gs_last_error() on failure."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise GsError(f"{name} failed (code {rc}): {lib.gs_last_error().decode(errors='replace')}")


def query(name, *args):
    return getattr(load(), name)(*args)


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


STAGE_NUM = 14
DEBUG_NO_BLOCK_CULL = 1
DEBUG_BWD_TILE = 2       # gs_render_backward: round 1's tile-parallel kernel instead of the segment-parallel one
DEBUG_FWD_HALFWARP = 4   # gs_render_forward: round 1's half-warp blend kernel instead of the packed two-pixel one
DEBUG_XR_PACK_CTA = 8    # direct exchange: CTA-compacted pack kernel (A/B switch)
DEBUG_BWD_SEG_R2 = 16    # gs_render_backward: round 2's segment-parallel kernel instead of round 3's (A/B switch)


def debug_set(flags):
    """Test-only switches (include/grendel_gs_b200.h, gs_debug_set); returns the previous flags."""
    return query("gs_debug_set", int(flags))


def profile_enable(on=True):
    call("gs_profile_enable", 1 if on else 0)


def profile_read():
    """-> {stage name: (total ms, launches)} for every stage that recorded launches; resets the counters."""
    out = {}
    for st in range(STAGE_NUM):
        ms, n = C.c_double(0.0), C.c_int64(0)
        call("gs_profile_read", st, C.byref(ms), C.byref(n))
        if n.value:
            out[load().gs_profile_stage_name(st).decode()] = (ms.value, n.value)
    return out
