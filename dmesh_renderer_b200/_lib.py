"""ctypes binding of libdmesh_b200.so (include/dmesh_b200.h).

The library is the product; there is no CPU or PyTorch fallback.  If the
shared object is missing, loading fails loudly.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# DMESH_B200_LIB: development override -- load another build of the SAME library (e.g. an experiment variant built
# from a modified tree) instead of the in-tree one.  It is not a fallback: a missing file still raises.
LIB_PATH = os.environ.get("DMESH_B200_LIB") or os.path.join(_HERE, "libdmesh_b200.so")

c_int = ctypes.c_int
c_size_t = ctypes.c_size_t
c_void_p = ctypes.c_void_p

_lib = None

# name -> (restype, argtypes).  Kept in the order of include/dmesh_b200.h; the
# CPU test-suite checks that every symbol declared there is exported.
SIGNATURES = {
    "dmr_abi_version": (c_int, []),
    "dmr_last_error": (ctypes.c_char_p, []),
    "dmr_tri_state_bytes": (c_int, [c_int] * 5 + [ctypes.POINTER(c_size_t)]),
    "dmr_tet_state_bytes": (c_int, [c_int] * 6 + [ctypes.POINTER(c_size_t)]),
    "dmr_binning_bytes": (c_size_t, [c_size_t]),
    "dmr_wait_i32": (c_int, [c_void_p, ctypes.c_int32, c_void_p]),
    "dmr_tri_forward_bin": (c_int, [c_int] * 5 + [c_void_p] * 11 + [c_void_p]),
    "dmr_tri_depth_chain": (c_int, [c_int, c_int] + [c_void_p] * 5 + [c_void_p]),
    "dmr_tri_forward_render": (c_int, [c_int] * 6 + [c_void_p] * 9 + [c_void_p]),
    "dmr_tri_face_weights_bytes": (c_size_t, [c_int] * 2),
    "dmr_tri_forward_render_face_weights": (c_int, [c_int] * 6 + [c_void_p] * 11 + [c_void_p, c_size_t] + [c_void_p]),
    "dmr_tri_backward_workspace_bytes": (c_size_t, [c_int] * 3),
    "dmr_tri_backward": (c_int, [c_int] * 6 + [c_void_p] * 14 + [c_void_p, c_size_t] + [c_void_p]),
    "dmr_tri_backward_deterministic_bytes": (c_size_t, [c_int] * 3),
    "dmr_tri_backward_deterministic": (c_int, [c_int] * 6 + [c_void_p] * 14 + [c_void_p, c_size_t] + [c_void_p]),
    "dmr_tri_backward_camera_bytes": (c_size_t, [c_int] * 6),
    "dmr_tri_backward_camera": (c_int, [c_int] * 6 + [c_void_p] * 14 + [c_int] + [c_void_p] * 2 + [c_void_p, c_size_t] + [c_void_p]),
    "dmr_tri_backward_exact": (c_int, [c_int] * 6 + [c_void_p] * 14 + [c_int] + [c_void_p] * 2 + [c_void_p, c_size_t] + [c_void_p]),
    "dmr_tri_backward_alpha": (c_int, [c_int] * 6 + [c_void_p] * 14 + [c_int] * 2 + [c_void_p] * 3 + [c_void_p, c_size_t] + [c_void_p]),
    "dmr_tri_alpha": (c_int, [c_int] * 3 + [c_void_p] * 2 + [c_void_p]),
    "dmr_tri_background_grad_bytes": (c_size_t, [c_int]),
    "dmr_tri_background_grad": (c_int, [c_int] * 3 + [c_void_p] * 4 + [c_size_t] + [c_void_p]),
    "dmr_tri_depth_chain_camera_bytes": (c_size_t, [c_int] * 2),
    "dmr_tri_depth_chain_camera": (c_int, [c_int, c_int] + [c_void_p] * 8 + [c_size_t, c_void_p]),
    "dmr_tet_records_bytes": (c_size_t, [c_int]),
    "dmr_tet_build_records": (c_int, [c_int] * 3 + [c_void_p] * 6 + [c_void_p]),
    "dmr_tet_forward_bin": (c_int, [c_int] * 6 + [c_void_p] * 12 + [c_int] + [c_void_p] * 2),
    "dmr_tet_forward_render": (c_int, [c_int] * 8 + [c_void_p] * 14 + [c_void_p]),
    "dmr_tet_forward_render_views": (c_int, [c_int] * 9 + [c_void_p] * 14 + [c_void_p]),
    "dmr_tet_backward_workspace_bytes": (c_size_t, [c_int]),
    "dmr_tet_backward": (c_int, [c_int] * 7 + [c_void_p] * 14 + [c_void_p, c_size_t] + [c_void_p]),
    "dmr_tet_backward_deterministic_bytes": (c_size_t, [c_int] * 2),
    "dmr_tet_backward_deterministic": (c_int, [c_int] * 7 + [c_void_p] * 14 + [c_void_p, c_size_t] + [c_void_p]),
    "dmr_tet_backward_camera_bytes": (c_size_t, [c_int] * 6),
    "dmr_tet_backward_camera": (c_int, [c_int] * 7 + [c_void_p] * 14 + [c_int] + [c_void_p] * 2 + [c_void_p, c_size_t] + [c_void_p]),
    "dmr_tet_backward_vertex_bytes": (c_size_t, [c_int] * 7),
    "dmr_tet_backward_vertex": (c_int, [c_int] * 7 + [c_void_p] * 14 + [c_int] + [c_void_p] * 3 + [c_void_p, c_size_t] + [c_void_p]),
    "dmr_tet_backward_intensity_bytes": (c_size_t, [c_int] * 8),
    "dmr_tet_backward_intensity": (c_int, [c_int] * 7 + [c_void_p] * 14 + [c_int] + [c_void_p] * 4 + [c_void_p, c_size_t] + [c_void_p]),
    "dmr_tet_backward_alpha": (c_int, [c_int] * 7 + [c_void_p] * 14 + [c_int] + [c_void_p] * 5 + [c_void_p, c_size_t] + [c_void_p]),
    "dmr_tet_alpha": (c_int, [c_int] * 3 + [c_void_p] * 2 + [c_void_p]),
    "dmr_tet_background_grad_bytes": (c_size_t, [c_int]),
    "dmr_tet_background_grad": (c_int, [c_int] * 3 + [c_void_p] * 4 + [c_size_t] + [c_void_p]),
    "dmr_tet_face_weights_bytes": (c_size_t, [c_int] * 2),
    "dmr_tet_face_weights": (c_int, [c_int] * 7 + [c_void_p] * 8 + [c_void_p, c_size_t] + [c_void_p]),
    "dmr_debug_view": (c_int, [c_int] * 8 + [c_size_t, c_void_p, ctypes.POINTER(c_void_p), ctypes.POINTER(c_size_t)]),
    "dmr_nvls_allreduce_sum_f32_fused": (c_int, [c_void_p, c_size_t, c_int, c_int, c_void_p, c_void_p, ctypes.c_uint, c_void_p]),
    "dmr_camera_inverses": (c_int, [c_int, c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, c_void_p, ctypes.c_int64,
                                   ctypes.c_int64, ctypes.c_int64, c_void_p, c_void_p, c_void_p]),
    "dmr_launch_count": (ctypes.c_ulonglong, []),
    "dmr_debug_set_tet_trail_cap": (c_int, [c_int]),
    "dmr_debug_set_tet_first_split": (c_int, [c_int]),
    "dmr_profile_enable": (c_int, [c_int]),
    "dmr_profile_stage_count": (c_int, []),
    "dmr_profile_stage_name": (ctypes.c_char_p, [c_int]),
    "dmr_profile_read": (c_int, [ctypes.POINTER(ctypes.c_float)]),
    "dmr_sort_temp_bytes": (c_size_t, [c_size_t]),
    "dmr_sort_pairs": (c_int, [c_void_p] * 4 + [c_size_t, c_int, c_void_p, c_void_p]),
    "dmr_sort_pairs_u32": (c_int, [c_void_p] * 4 + [c_size_t, c_int, c_void_p, c_void_p]),
}


def load():
    """Load the native library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "dmesh_renderer_b200: native library %s not found. Build it with "
            "`python -m dmesh_renderer_b200.build` (needs nvcc, sm_100a). There is no fallback path." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().dmr_last_error()
        raise RuntimeError("libdmesh_b200: %s (code %d)" % (msg.decode() if msg else "error", rc))
