"""ctypes binding of libdatum_ibl_cuda (include/datum_ibl_cuda.h)."""

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# DATUM_IBL_CUDA_LIB: another build of the same C ABI (the tools build with the A/B kernel variants,
# tools/ab/libdatum_ibl_cuda_ab.so); never set by the product, the tests or the benchmark
LIB_PATH = os.environ.get("DATUM_IBL_CUDA_LIB") or os.path.join(_HERE, "lib", "libdatum_ibl_cuda.so")

_lib = None

c_void_p = ctypes.c_void_p
c_int = ctypes.c_int
c_float = ctypes.c_float
c_size_t = ctypes.c_size_t

# name -> (restype, argtypes); every symbol include/datum_ibl_cuda.h declares
SIGNATURES = {
    "datum_ibl_create": (c_int, [c_int, ctypes.POINTER(c_void_p)]),
    "datum_ibl_destroy": (None, [c_void_p]),
    "datum_ibl_last_error": (ctypes.c_char_p, []),
    "datum_ibl_stream": (c_void_p, [c_void_p]),
    "datum_ibl_synchronize": (c_int, [c_void_p]),
    "datum_ibl_launch_count": (ctypes.c_uint64, [c_void_p]),
    "datum_ibl_set_prefilter_variant": (c_int, [c_void_p, c_int]),
    "datum_ibl_set_tuning": (c_int, [c_void_p, ctypes.c_char_p, c_int]),
    "datum_ibl_chain_bytes": (c_size_t, [c_int, c_int, c_int]),
    "datum_ibl_buildmips_cube_ibl": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "datum_ibl_bake_probes": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_void_p), c_void_p]),
    "datum_ibl_buildmips_cube_ibl_device": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "datum_ibl_prefilter_level_device": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "datum_ibl_prefilter_level_peers": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p), ctypes.c_uint32]),
    "datum_ibl_peer_barrier": (c_int, [c_void_p, c_int, c_int, ctypes.POINTER(c_void_p), ctypes.c_uint32]),
    "datum_ibl_set_peer_timeout_ms": (c_int, [c_void_p, c_int]),
    "datum_ibl_peer_alloc": (c_int, [c_void_p, c_size_t, ctypes.POINTER(c_void_p), c_void_p]),
    "datum_ibl_peer_free": (c_int, [c_void_p, c_void_p]),
    "datum_ibl_peer_open": (c_int, [c_void_p, c_void_p, ctypes.POINTER(c_void_p)]),
    "datum_ibl_peer_close": (c_int, [c_void_p, c_void_p]),
    "datum_ibl_multi_create": (c_int, [c_int, ctypes.POINTER(c_int), ctypes.POINTER(c_void_p)]),
    "datum_ibl_multi_destroy": (None, [c_void_p]),
    "datum_ibl_multi_device_count": (c_int, [c_void_p]),
    "datum_ibl_multi_context": (c_void_p, [c_void_p, c_int]),
    "datum_ibl_multi_buildmips_cube_ibl": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "datum_ibl_multi_bake_probes": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_void_p), c_void_p]),
    "datum_ibl_multi_project_sh9": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "datum_ibl_buildmips_cube_ibl_devices": (c_int, [c_int, ctypes.POINTER(c_int), c_int, c_int, c_int, c_int, c_void_p]),
    "datum_ibl_bake_probes_devices": (c_int, [c_int, ctypes.POINTER(c_int), c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_void_p), c_void_p]),
    "datum_ibl_sh9_partial_device": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "datum_ibl_sh9_partial_peers": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p), ctypes.c_uint32]),
    "datum_ibl_sh9_finish": (None, [c_void_p, c_void_p]),
    "datum_ibl_project_sh9": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "datum_ibl_sh9_irradiance_cube": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "datum_ibl_pack_envbrdf": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p]),
    "datum_ibl_pack_watercolor": (c_int, [c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_float, c_float, c_int, c_int, c_void_p]),
    "datum_ibl_pack_cube_ibl": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "datum_ibl_pack_cube": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_void_p]),
    "datum_ibl_ingest_cube_argb32": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "datum_ibl_ingest_cube_argb32_ibl": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "datum_ibl_measure_fp32_peak": (c_int, [c_void_p, ctypes.POINTER(ctypes.c_double)]),
    "datum_ibl_measure_fp32x2_peak": (c_int, [c_void_p, ctypes.POINTER(ctypes.c_double)]),
    "datum_ibl_dominant_kernel_stats": (c_int, [c_void_p, c_int, ctypes.POINTER(c_int), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]),
    "datum_ibl_last_prefilter_ms": (c_int, [c_void_p, ctypes.POINTER(c_float)]),
    "datum_ibl_buildmips_cube_float": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "datum_ibl_buildmips_cube_float_device": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "datum_ibl_prefilter_level_float_device": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "datum_ibl_bake_probes_float": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_void_p), c_void_p]),
    "datum_ibl_multi_bake_probes_float": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_void_p), c_void_p]),
}


def load():
    """Load the CUDA library; fail loudly if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libdatum_ibl_cuda.so is missing (%s): run `python -m datum_b200.build`. "
                "datum_b200 has no CPU fallback." % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the header and the library disagree
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = lib
    return _lib
