"""ctypes loader for libdang_gpu.so (the C ABI of include/dang_gpu.h).

There is no fallback: if the shared library is missing or cannot be loaded this raises, and if
no CUDA device is present `dang_gpu_create` returns an error that `Engine` turns into an
exception.  The library is built in-tree by dang_b200/csrc/build.sh (see __graft_entry__.build).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdang_gpu.so")

c_dp = C.POINTER(C.c_double)
c_ip = C.POINTER(C.c_int)
c_i64p = C.POINTER(C.c_int64)
vp = C.c_void_p

# every symbol include/dang_gpu.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "dang_gpu_create": (C.c_int, [C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int64,
                                  C.c_int64, C.POINTER(vp)]),
    "dang_gpu_destroy": (C.c_int, [vp]),
    "dang_gpu_last_error": (C.c_char_p, [vp]),
    "dang_gpu_set_option": (C.c_int, [vp, C.c_int, C.c_double]),
    "dang_gpu_sync": (C.c_int, [vp]),
    "dang_gpu_comm_unique_id": (C.c_int, [C.c_char_p]),
    "dang_gpu_comm_init": (C.c_int, [vp, C.c_int, C.c_int, C.c_char_p]),
    "dang_gpu_comm_ipc_handle": (C.c_int, [vp, C.c_char_p]),
    "dang_gpu_comm_open_peers": (C.c_int, [vp, C.c_char_p]),
    "dang_gpu_comm_check": (C.c_int, [vp]),
    "dang_gpu_set_band": (C.c_int, [vp, C.c_int, C.c_double, C.c_int, c_dp, c_dp]),
    "dang_gpu_upload_maps": (C.c_int, [vp, c_dp, c_dp, c_dp, c_dp, c_dp]),
    "dang_gpu_share_maps": (C.c_int, [vp, vp]),
    "dang_gpu_set_gain_offset": (C.c_int, [vp, c_dp, c_dp]),
    "dang_gpu_set_component": (C.c_int, [vp, C.c_int, C.c_int, C.c_char_p, C.c_double, C.c_int, C.c_int,
                                         c_dp, c_dp]),
    "dang_gpu_set_template": (C.c_int, [vp, C.c_int, c_dp, c_dp, c_ip, C.c_int]),
    "dang_gpu_get_template_amplitudes": (C.c_int, [vp, C.c_int, c_dp]),
    "dang_gpu_set_index": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_dp, c_dp,
                                     C.c_double, C.c_int, c_ip, C.c_int]),
    "dang_gpu_set_amplitude": (C.c_int, [vp, C.c_int, c_dp]),
    "dang_gpu_set_indices": (C.c_int, [vp, C.c_int, c_dp]),
    "dang_gpu_get_amplitude": (C.c_int, [vp, C.c_int, c_dp]),
    "dang_gpu_get_indices": (C.c_int, [vp, C.c_int, c_dp]),
    "dang_gpu_get_index_fullsky": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, c_dp]),
    "dang_gpu_get_step_size": (C.c_int, [vp, C.c_int, C.c_int, c_dp]),
    "dang_gpu_set_cg_group": (C.c_int, [vp, C.c_int, C.c_int, C.c_double, c_ip, C.c_int]),
    "dang_gpu_cg_solve": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, c_dp, C.c_uint64, c_ip, c_dp]),
    "dang_gpu_cg_trace": (C.c_int, [vp, c_dp, C.c_int, c_ip]),
    "dang_gpu_get_cg_x": (C.c_int, [vp, C.c_int, C.c_int, c_dp]),
    "dang_gpu_sample_index": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_dp, c_dp,
                                        C.c_uint64, c_dp]),
    "dang_gpu_get_decisions": (C.c_int, [vp, C.POINTER(C.c_ubyte), c_dp]),
    "dang_gpu_perpixel_stats": (C.c_int, [vp, c_dp, c_dp]),
    "dang_gpu_tune_index": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_dp, c_dp,
                                      C.c_uint64, C.c_int, c_ip, c_dp]),
    "dang_gpu_chisq": (C.c_int, [vp, C.c_int, C.c_int, c_dp, c_i64p]),
    "dang_gpu_get_sky_model": (C.c_int, [vp, C.c_int, C.c_int, c_dp, c_dp, c_dp]),
    "dang_gpu_fit_band_gain": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, c_dp, C.c_uint64, c_dp]),
    "dang_gpu_index_mean": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, c_dp]),
    "dang_gpu_iteration_mark": (C.c_int, [vp, C.POINTER(C.c_int64)]),
    "dang_gpu_iteration_scalars": (C.c_int, [vp, C.c_int64, C.POINTER(C.c_int), c_dp, c_dp, c_dp, c_dp, c_dp]),
    "dang_gpu_get_amplitude_async": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, c_dp]),
    "dang_gpu_get_indices_async": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, c_dp]),
    "dang_gpu_download_wait": (C.c_int, [vp]),
    "dang_gpu_stage_eta": (C.c_int, [vp, c_dp, C.c_int]),
    "dang_gpu_bandpass_quadrature": (C.c_int, [C.c_double, C.c_int, c_dp, c_dp, C.c_int, c_dp, c_dp]),
    "dang_gpu_band_samples": (C.c_int, [vp, C.c_int, c_ip]),
    "dang_gpu_host_alloc": (C.c_int, [C.POINTER(vp), C.c_uint64]),
    "dang_gpu_host_free": (C.c_int, [vp]),
    "dang_gpu_event_record": (C.c_int, [vp, C.c_int]),
    "dang_gpu_event_elapsed_ms": (C.c_int, [vp, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    "dang_gpu_launch_count": (C.c_int, [vp, c_i64p, C.c_int]),
    "dang_gpu_kernel_stats": (C.c_int, [vp, C.c_int, c_i64p, c_dp, c_dp, C.c_int]),
    "dang_gpu_kernel_name": (C.c_char_p, [C.c_int]),
    "dang_gpu_timeline": (C.c_int, [vp, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), c_dp, c_dp]),
    "dang_gpu_set_t_cmb": (C.c_int, [vp, C.c_double]),
    "dang_gpu_udgrade": (C.c_int, [vp, C.c_int, c_dp, C.c_int, c_dp, C.c_int, C.c_int, C.c_double]),
    "dang_gpu_comm_probe": (C.c_int, [vp, C.c_int, C.c_int, c_dp]),
    "dang_gpu_posterior_begin": (C.c_int, [vp, C.c_int, C.c_int, C.c_int]),
    "dang_gpu_posterior_accumulate": (C.c_int, [vp]),
    "dang_gpu_posterior_get": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, c_dp, c_dp, c_i64p]),
    "dang_gpu_posterior_end": (C.c_int, [vp]),
    "dang_gpu_posterior_rhat": (C.c_int, [C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_int, c_dp]),
    "dang_gpu_posterior_begin_batched": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int]),
    "dang_gpu_posterior_ess": (C.c_int, [C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_int, c_dp, c_dp]),
}

_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with dang_b200/csrc/build.sh "
            "(__graft_entry__.build()).  dang_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export the symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
