"""ctypes binding of libfslic_b200.so (the C ABI declared in include/fslic_b200.h).

The library is built in-tree by ``fast_slic_b200/csrc/build.sh`` (see ``__graft_entry__.build``).
There is no CPU fallback: if the shared library is missing the import fails loudly.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfslic_b200.so")

# every symbol include/fslic_b200.h declares
EXPORTED_SYMBOLS = (
    "fslic_b200_last_error", "fslic_b200_version", "fslic_b200_sizeof_cluster", "fslic_b200_create",
    "fslic_b200_destroy", "fslic_b200_initialize_clusters", "fslic_b200_iterate", "fslic_b200_iterate_host",
    "fslic_b200_initialize_clusters_host", "fslic_b200_enforce_connectivity", "fslic_b200_debug_stages",
    "fslic_b200_rgb_to_quad", "fslic_b200_debug_heap_select", "fslic_b200_stage_ms", "fslic_b200_get_S",
    "fslic_b200_launches_last_iterate", "fslic_b200_assign_kernel_time", "fslic_b200_debug_cca_counters", "fslic_b200_debug_select_profile",
    "fslic_b200_iterate_host_async", "fslic_b200_wait", "fslic_b200_create_cca",
    "fslic_b200_debug_assign_impl", "fslic_b200_connectivity_scratch_bytes", "fslic_b200_get_connectivity",
    "fslic_b200_get_mask_density", "fslic_b200_cluster_density_to_mask", "fslic_b200_cca_stage_ms",
    "fslic_b200_iterate_real", "fslic_b200_iterate_preemptive", "fslic_b200_set_manhattan_spatial_dist",
)

STAGE_NAMES = ("cielab_conversion", "assign", "update", "full_assign", "enforce_connectivity", "iterate")
CCA_STAGE_NAMES = ("build_disjoint_set", "flatten", "threshold_by_area", "sort", "substitute", "output")  # cca.cpp:194-263


class Params(C.Structure):
    """== fslic_params (include/fslic_b200.h)."""
    _fields_ = [("compactness", C.c_float), ("min_size_factor", C.c_float), ("subsample_stride", C.c_int32),
                ("convert_to_lab", C.c_int32), ("max_iter", C.c_int32), ("collect_timing", C.c_int32)]


class FslicError(RuntimeError):
    pass


_lib = None


def build_library(verbose=False):
    import subprocess
    script = os.path.join(_HERE, "csrc", "build.sh")
    subprocess.check_call(["bash", script], stdout=None if verbose else subprocess.DEVNULL)


def lib():
    """Load (once) and return the C-ABI library."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "fast_slic_b200: %s is missing -- build it with fast_slic_b200/csrc/build.sh "
            "(there is no CPU fallback)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i32 = C.c_void_p, C.c_int
    L.fslic_b200_last_error.restype = C.c_char_p
    L.fslic_b200_version.restype = C.c_char_p
    L.fslic_b200_create.argtypes = [i32, i32, i32, i32, i32, C.POINTER(vp)]
    L.fslic_b200_create_cca.argtypes = [i32, i32, i32, i32, C.POINTER(vp)]
    L.fslic_b200_destroy.argtypes = [vp]
    L.fslic_b200_initialize_clusters.argtypes = [vp, vp, vp, i32, vp]
    L.fslic_b200_iterate.argtypes = [vp, vp, vp, vp, i32, C.POINTER(Params), vp]
    L.fslic_b200_iterate_real.argtypes = [vp, i32, vp, vp, vp, i32, C.POINTER(Params), vp]
    L.fslic_b200_iterate_preemptive.argtypes = [vp, vp, vp, vp, i32, C.POINTER(Params), C.c_float, vp]
    L.fslic_b200_iterate_host.argtypes = [vp, vp, vp, vp, i32, C.POINTER(Params)]
    L.fslic_b200_iterate_host_async.argtypes = [vp, vp, vp, vp, i32, C.POINTER(Params)]
    L.fslic_b200_wait.argtypes = [vp]
    L.fslic_b200_initialize_clusters_host.argtypes = [vp, vp, vp, i32]
    L.fslic_b200_enforce_connectivity.argtypes = [vp, vp, i32, i32, i32, vp]
    L.fslic_b200_debug_stages.argtypes = [vp, vp, vp, i32, vp]
    L.fslic_b200_rgb_to_quad.argtypes = [vp, vp, vp, i32, i32, vp]
    L.fslic_b200_debug_heap_select.argtypes = [vp, vp, i32, i32, vp, vp]
    L.fslic_b200_stage_ms.argtypes = [vp, C.POINTER(C.c_float), i32]
    L.fslic_b200_cca_stage_ms.argtypes = [vp, C.POINTER(C.c_float), i32]
    L.fslic_b200_get_S.argtypes = [vp]
    L.fslic_b200_launches_last_iterate.argtypes = [vp]
    L.fslic_b200_debug_assign_impl.argtypes = [vp]
    L.fslic_b200_set_manhattan_spatial_dist.argtypes = [vp, i32]
    L.fslic_b200_connectivity_scratch_bytes.argtypes = [i32]
    L.fslic_b200_connectivity_scratch_bytes.restype = C.c_size_t
    L.fslic_b200_get_connectivity.argtypes = [i32, i32, i32, i32, vp, vp, vp, vp, C.c_size_t, vp]
    L.fslic_b200_get_mask_density.argtypes = [i32, i32, i32, i32, vp, vp, vp, vp, vp, vp]
    L.fslic_b200_cluster_density_to_mask.argtypes = [i32, i32, i32, i32, vp, vp, vp, vp]
    L.fslic_b200_assign_kernel_time.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_int)]
    L.fslic_b200_debug_cca_counters.argtypes = [vp, C.POINTER(C.c_int32), i32]
    L.fslic_b200_debug_select_profile.argtypes = [vp, C.POINTER(C.c_longlong), i32]
    assert L.fslic_b200_sizeof_cluster() == 32
    _lib = L
    return L


def check(rc):
    if rc != 0:
        msg = lib().fslic_b200_last_error().decode("utf-8", "replace")
        if rc == -1:
            raise ValueError(msg)
        if rc == -3:
            raise MemoryError(msg)
        raise FslicError("fslic_b200 error %d: %s" % (rc, msg))
