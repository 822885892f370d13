"""ctypes binding of libsitrack_b200.so (the C ABI in include/sitrack_b200.h).

There is no CPU fallback: if the library is missing or no CUDA device is
present every compute entry point raises `SitrackCudaError`.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("SITRACK_B200_LIB") or os.path.join(HERE, "libsitrack_b200.so")   # env: A/B builds

ST_OK, ST_EINVAL, ST_ECUDA, ST_ESTATE, ST_ENOMEM = 0, -1, -2, -3, -4


class SitrackCudaError(RuntimeError):
    pass


_lib = None

c_i64, c_int, c_dbl, vp = C.c_int64, C.c_int, C.c_double, C.c_void_p

# name -> (restype, argtypes); every symbol declared in include/sitrack_b200.h
SIGNATURES = {
    "st_abi_version": (c_int, []),
    "st_last_error": (C.c_char_p, [vp]),
    "st_create": (c_int, [C.POINTER(vp), c_int, c_int, c_int] + [vp] * 7 + [c_int, c_dbl, c_dbl]),
    "st_destroy": (None, [vp]),
    "st_set_projection": (c_int, [vp, c_dbl, c_dbl]),
    "st_set_kernel_variant": (c_int, [vp, c_int]),
    "st_selftest_xy2latlon_fast": (c_int, [c_int, c_i64, vp, vp, c_dbl, c_dbl]),
    "st_selftest_proj": (c_int, [c_int, c_int, c_i64, vp, vp, c_dbl, c_dbl, c_dbl, c_dbl]),
    "st_selftest_div1000": (c_int, [c_int, c_i64, vp, vp, vp]),
    "st_selftest_divide": (c_int, [c_int, c_i64, vp, vp, vp, vp]),
    "st_cert_stats": (c_int, [vp, C.POINTER(c_i64), C.POINTER(c_i64)]),
    "st_cert_frames": (c_int, [vp, vp, vp]),
    "st_selftest_cert": (c_int, [vp, c_i64, vp, vp, vp, vp]),
    "st_set_locate_grid": (c_int, [vp, vp, vp, vp]),
    "st_seed_locate": (c_int, [vp, c_i64, vp, vp, vp, vp, vp, vp]),
    "st_seed_compact_dev": (c_int, [vp, c_i64, vp, vp, vp, vp, vp, C.POINTER(c_i64), vp]),
    "st_seed_locate_ex": (c_int, [vp, c_i64, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "st_seed_locate_dev": (c_int, [vp, c_i64, vp, vp, vp, vp, vp, vp, vp]),
    "st_nearest_point": (c_int, [vp, c_i64, vp, c_dbl, c_int, c_int, vp, vp]),
    "st_find_containing_cell": (c_int, [vp, c_i64, vp, vp, vp, vp]),
    "st_set_buoys": (c_int, [vp, c_i64, vp, vp, vp, vp]),
    "st_set_buoys_dev": (c_int, [vp, c_i64, vp, vp, vp, vp, vp]),
    "st_get_state": (c_int, [vp, vp, vp, vp]),
    "st_state_device_ptrs": (c_int, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]),
    "st_set_row_chain": (c_int, [vp, c_int]),
    "st_sync_state": (c_int, [vp, vp]),
    "st_num_buoys": (c_i64, [vp]),
    "st_record_slots": (c_int, [vp, c_int]),
    "st_record_host_buffer": (c_int, [vp, c_int, C.POINTER(vp)]),
    "st_record_device_buffer": (c_int, [vp, c_int, C.POINTER(vp)]),
    "st_submit_record": (c_int, [vp, c_int, vp]),
    "st_upload_record": (c_int, [vp, c_int, vp, vp]),
    "st_step": (c_int, [vp, c_int, c_int, vp, vp, vp, vp, vp]),
    "st_step_multi": (c_int, [vp, vp, c_i64, c_int, c_int, vp, vp, vp, c_i64, vp, vp]),
    "st_track_record_host": (c_int, [vp, c_int, vp, vp, vp, vp, vp, vp, C.POINTER(c_i64)]),
    "st_step_ext": (c_int, [vp, c_int, c_int, c_int, c_int, c_int, vp, vp, vp, vp, vp]),
    "st_step_f4": (c_int, [vp, c_int, c_int, vp, vp, vp, vp, vp]),
    "st_step_multi_f4": (c_int, [vp, vp, c_i64, c_int, c_int, vp, vp, vp, c_i64, vp, vp]),
    "st_track_record_host_f4": (c_int, [vp, c_int, vp, vp, vp, vp, vp, vp, C.POINTER(c_i64)]),
    "st_gather_create": (c_int, [vp, c_int, c_int, c_i64, c_i64, c_int, c_int, vp]),
    "st_gather_connect_ipc": (c_int, [vp, vp]),
    "st_gather_connect_ptrs": (c_int, [vp, C.POINTER(vp)]),
    "st_gather_block": (c_int, [vp, C.POINTER(vp), C.POINTER(c_i64)]),
    "st_gather_buffer": (c_int, [vp, c_int, C.POINTER(vp)]),
    "st_step_gather": (c_int, [vp, c_int, c_int, c_int, C.c_uint64, vp, vp, vp, vp]),
    "st_gather_wait": (c_int, [vp, C.c_uint64, vp]),
    "st_gather_ack": (c_int, [vp, C.c_uint64, vp]),
    "st_gather_timed_out": (c_int, [vp, C.POINTER(c_int)]),
    "st_gather_destroy": (c_int, [vp]),
    "st_gather_set_mode": (c_int, [vp, c_int]),
    "st_deform_dev": (c_int, [vp, c_i64, vp, vp, vp, vp, vp, c_dbl, vp, vp]),
    "st_deform_scales_scratch_bytes": (c_int, [c_i64, c_int, vp, vp, c_int, vp]),
    "st_deform_scales_dev": (c_int, [vp, c_i64, vp, vp, vp, vp, vp, c_dbl, c_int, vp, vp, vp, vp, c_int, vp, vp, c_i64,
                                     vp, vp, vp, vp]),
    "st_deform_grid_scratch_bytes": (c_int, [c_i64, c_int, c_int, c_int, c_int, vp]),
    "st_deform_grid_dev": (c_int, [vp, c_i64, vp, vp, vp, vp, vp, c_dbl, c_int, c_int, c_int, c_dbl, c_dbl, c_dbl, vp,
                                   c_int, vp, vp, c_i64, vp, vp, vp, vp, vp]),
    "st_deform_grid_stages_dev": (c_int, [vp, c_i64, vp, vp, vp, vp, vp, c_dbl, c_int, c_int, c_int, c_dbl, c_dbl, c_dbl,
                                          vp, c_int, vp, vp, c_i64, vp, vp, vp, vp, c_int, vp]),
    "st_dispersion_scratch_bytes": (c_int, [c_i64, c_int, c_int, c_int, vp]),
    "st_dispersion_dev": (c_int, [vp, c_i64, vp, vp, vp, c_int, vp, vp, vp, c_dbl, c_int, c_int, vp, c_int, vp, vp,
                                  c_i64, vp, vp, vp, vp]),
    "st_fsle_state_bytes": (c_int, [c_i64, c_int, c_int, vp]),
    "st_fsle_dev": (c_int, [vp, c_i64, vp, vp, vp, vp, c_int, vp, vp, c_int, vp, c_int, vp, vp, vp]),
    "st_sample_dev": (c_int, [vp, c_int, vp, c_i64, vp, vp, c_int, vp, vp, vp]),
    "st_xy2latlon": (c_int, [c_int, c_i64, vp, vp, c_dbl, c_dbl]),
    "st_latlon2xy": (c_int, [c_int, c_i64, vp, vp, c_dbl, c_dbl]),
    "st_xy2latlon_dev": (c_int, [c_i64, vp, vp, c_dbl, c_dbl, vp]),
    "st_intersect2seg": (c_int, [c_int, c_i64, vp, vp, vp, vp, vp]),
    "st_inside_quad": (c_int, [c_int, c_i64, vp, vp, vp]),
    "st_cell_walk": (c_int, [c_int, c_i64, vp, vp, vp, vp, vp, vp]),
    "st_survive": (c_int, [c_int, c_i64, vp, c_int, c_int, vp, vp, c_dbl, vp]),
    "st_haversine": (c_int, [c_int, c_i64, c_dbl, c_dbl, vp, vp, vp]),
}


def lib():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise SitrackCudaError(
                "libsitrack_b200.so is not built (run `python -m sitrack_b200.build`); "
                "sitrack_b200 has no CPU fallback")
        L = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(L, name)
            f.restype, f.argtypes = res, args
        if L.st_abi_version() != 3:
            raise SitrackCudaError("libsitrack_b200.so ABI version mismatch")
        _lib = L
    return _lib


def check(rc, ctx=None):
    if rc != ST_OK:
        msg = lib().st_last_error(ctx)
        raise SitrackCudaError("libsitrack_b200 error %d: %s" % (rc, (msg or b"").decode()))


def hptr(a):
    """Pointer of a C-contiguous numpy array (None -> NULL)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data


def as_c(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)
