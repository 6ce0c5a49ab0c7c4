"""ctypes binding of the C ABI in include/gmpi_mpi_render.h.

There is no CPU or PyTorch fallback: if the library is missing or fails to load this raises."""
import ctypes
import os

from ._build import LIB_PATH

GMPI_OK = 0
FLAG_RGBA_RANGE = 1
FLAG_ALPHA_RANGE = 2
FLAG_LAST_PLANE_OOB = 4
FLAG_PLANE_BEHIND_EYE = 8

OPT_ALIGN_CORNERS = 1
OPT_CHECK_LAST_PLANE = 2
OPT_COLOR_MINUS1_1 = 4
OPT_ZERO_GRAD = 8

PLAN_DIRECT, PLAN_STAGED = 1, 2
WHY = {1: "texture width is not a multiple of 4", 2: "fewer than 120 tiles of 64x30 pixels", 4: "more than 512 planes",
       8: "rgba base pointer not 16-byte aligned", 16: "direct kernel forced by gmpi_debug_set_fwd_variant"}

ABI_VERSION = 2

EXPORTS = [
    "gmpi_abi_version", "gmpi_last_error", "gmpi_mpi_render_fwd_variant", "gmpi_mpi_render_fwd",
    "gmpi_mpi_render_fwd_gather", "gmpi_mpi_render_fwd_train", "gmpi_mpi_render_bwd", "gmpi_mpi_render_bwd_saved", "gmpi_mpi_check_range", "gmpi_mpi_render_fwd_host", "gmpi_mpi_release_host_cache", "gmpi_debug_plane_coords", "gmpi_debug_division", "gmpi_debug_set_fwd_variant", "gmpi_debug_set_bwd_zero", "gmpi_debug_copy_plan", "gmpi_debug_plane_coords_packed", "gmpi_debug_tile_walk",
    "gmpi_mpi_render_fwd_plan", "gmpi_mpi_render_fwd_ex", "gmpi_mpi_render_bwd_ex", "gmpi_mpi_render_host_ex",
    "gmpi_debug_tile_walk_ex", "gmpi_debug_cam_rays",
    "gmpi_mpi_zero_async", "gmpi_mpi_alpha_depth_fwd", "gmpi_mpi_alpha_depth_bwd", "gmpi_mpi_apply_shading_fwd", "gmpi_mpi_apply_shading_bwd",
    "gmpi_mpi_occupancy_plane_words", "gmpi_mpi_occupancy", "gmpi_mpi_render_fwd_skip_ex",
]

OPT_U8_ROUND_HALF_UP = 16


class RenderDesc(ctypes.Structure):
    """gmpi_render_desc of include/gmpi_mpi_render.h (field for field)."""
    _fields_ = [("struct_bytes", ctypes.c_uint32), ("options", ctypes.c_uint32),
                ("M", ctypes.c_int32), ("V", ctypes.c_int32), ("N", ctypes.c_int32), ("Ht", ctypes.c_int32), ("Wt", ctypes.c_int32),
                ("H", ctypes.c_int32), ("W", ctypes.c_int32), ("view_group", ctypes.c_int32),
                ("n_peers", ctypes.c_int32), ("frame_offset", ctypes.c_int32),
                ("depth_near", ctypes.c_float), ("depth_range", ctypes.c_float)] + \
               [(n, ctypes.c_void_p) for n in ("rgba", "rgb", "alpha", "bg_rgb", "view2mpi", "dhw", "ray_dir", "eye", "z_dir", "cam",
                                               "color", "depth", "transmittance", "peer_frames", "video_rgb", "video_depth",
                                               "g_color", "g_depth", "g_rgba", "g_rgb", "g_bg_rgb", "g_alpha", "flags", "stream")] + \
               [("stop_transmittance", ctypes.c_float), ("skipped_pixel_planes", ctypes.c_void_p)]     # appended (early termination)


# struct_bytes of the descriptor before the early-termination fields: still accepted, the fields then read as absent
DESC_BYTES_WITHOUT_STOP = RenderDesc.stop_transmittance.offset


def make_desc(**kw) -> RenderDesc:
    """RenderDesc with struct_bytes set; tensors are passed as such (their data_ptr is taken), None -> NULL."""
    d = RenderDesc()
    d.struct_bytes = ctypes.sizeof(RenderDesc)
    for k, v in kw.items():
        if v is None:
            continue
        if hasattr(v, "data_ptr"):
            v = v.data_ptr()
        setattr(d, k, v)
    return d


_lib = None


class GmpiLibraryError(RuntimeError):
    pass


def load():
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("GMPI_LIB_PATH", LIB_PATH)     # override: A/B-testing kernel builds
    if not os.path.exists(path):
        raise GmpiLibraryError(
            f"{path} is missing: the CUDA (sm_100a) renderer is not built. Run "
            "`python -c 'import __graft_entry__ as g; g.build()'` (needs nvcc). There is no CPU fallback.")
    lib = ctypes.CDLL(path)
    vp, i, u32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint32
    lib.gmpi_abi_version.restype = i
    lib.gmpi_abi_version.argtypes = []
    lib.gmpi_last_error.restype = ctypes.c_char_p
    lib.gmpi_last_error.argtypes = []
    lib.gmpi_mpi_render_fwd_variant.restype = ctypes.c_char_p
    lib.gmpi_mpi_render_fwd_variant.argtypes = [i] * 5
    lib.gmpi_mpi_render_fwd_plan.restype = i
    lib.gmpi_mpi_render_fwd_plan.argtypes = [i] * 6 + [vp, vp]
    lib.gmpi_mpi_render_fwd.restype = i
    lib.gmpi_mpi_render_fwd.argtypes = [vp] * 9 + [i] * 7 + [u32, vp]
    lib.gmpi_mpi_render_fwd_gather.restype = i
    lib.gmpi_mpi_render_fwd_gather.argtypes = [vp] * 7 + [i, i, vp] + [i] * 7 + [u32, vp]
    lib.gmpi_mpi_render_fwd_train.restype = i
    lib.gmpi_mpi_render_fwd_train.argtypes = [vp] * 10 + [i] * 7 + [u32, vp]
    lib.gmpi_mpi_render_bwd_saved.restype = i
    lib.gmpi_mpi_render_bwd_saved.argtypes = [vp] * 10 + [i] * 7 + [u32, vp]
    lib.gmpi_mpi_render_bwd.restype = i
    lib.gmpi_mpi_render_bwd.argtypes = [vp] * 9 + [i] * 7 + [u32, vp]
    lib.gmpi_mpi_check_range.restype = i
    lib.gmpi_mpi_check_range.argtypes = [vp, i, i, i, i, vp, vp]
    lib.gmpi_mpi_render_fwd_host.restype = i
    lib.gmpi_mpi_render_fwd_host.argtypes = [vp] * 9 + [i] * 7 + [u32, i]
    lib.gmpi_mpi_release_host_cache.restype = i
    lib.gmpi_mpi_release_host_cache.argtypes = []
    lib.gmpi_debug_plane_coords.restype = i
    lib.gmpi_debug_plane_coords.argtypes = [vp] * 5 + [i] * 6 + [u32, vp]
    lib.gmpi_debug_plane_coords_packed.restype = i
    lib.gmpi_debug_plane_coords_packed.argtypes = [vp] * 5 + [i] * 6 + [u32, vp]
    lib.gmpi_debug_division.restype = i
    lib.gmpi_debug_division.argtypes = [vp, vp, vp, vp, ctypes.c_size_t, vp]
    lib.gmpi_debug_set_fwd_variant.restype = i
    lib.gmpi_debug_set_fwd_variant.argtypes = [i]
    lib.gmpi_debug_set_bwd_zero.restype = i
    lib.gmpi_debug_set_bwd_zero.argtypes = [i]
    lib.gmpi_debug_copy_plan.restype = i
    lib.gmpi_debug_copy_plan.argtypes = [i, vp, i]
    lib.gmpi_debug_tile_walk.restype = i
    lib.gmpi_debug_tile_walk.argtypes = [i, i, i, i, i, vp, i]
    lib.gmpi_debug_tile_walk_ex.restype = i
    lib.gmpi_debug_tile_walk_ex.argtypes = [i, i, i, i, i, i, i, vp, i]
    lib.gmpi_debug_cam_rays.restype = i
    lib.gmpi_debug_cam_rays.argtypes = [vp, vp, i, i, i, vp]
    for fn in (lib.gmpi_mpi_render_fwd_ex, lib.gmpi_mpi_render_bwd_ex):
        fn.restype = i
        fn.argtypes = [ctypes.POINTER(RenderDesc)]
    lib.gmpi_mpi_zero_async.restype = i
    lib.gmpi_mpi_zero_async.argtypes = [vp, ctypes.c_size_t, vp]
    ll = ctypes.c_longlong
    lib.gmpi_mpi_alpha_depth_fwd.restype = i
    lib.gmpi_mpi_alpha_depth_fwd.argtypes = [vp, ll, ll, vp, vp, vp, i, i, i, i, vp]
    lib.gmpi_mpi_alpha_depth_bwd.restype = i
    lib.gmpi_mpi_alpha_depth_bwd.argtypes = [vp, ll, ll, vp, vp, vp, vp, ll, ll, i, i, i, i, vp]
    lib.gmpi_mpi_apply_shading_fwd.restype = i
    lib.gmpi_mpi_apply_shading_fwd.argtypes = [vp, vp, vp, i, i, i, i, vp]
    lib.gmpi_mpi_apply_shading_bwd.restype = i
    lib.gmpi_mpi_apply_shading_bwd.argtypes = [vp, vp, vp, vp, vp, i, i, i, i, vp]
    lib.gmpi_mpi_render_host_ex.restype = i
    lib.gmpi_mpi_render_host_ex.argtypes = [ctypes.POINTER(RenderDesc), i]
    lib.gmpi_mpi_occupancy_plane_words.restype = ctypes.c_size_t
    lib.gmpi_mpi_occupancy_plane_words.argtypes = [i, i]
    lib.gmpi_mpi_occupancy.restype = i
    lib.gmpi_mpi_occupancy.argtypes = [vp, ll, ll, i, i, i, i, ctypes.c_float, vp, vp]
    lib.gmpi_mpi_render_fwd_skip_ex.restype = i
    lib.gmpi_mpi_render_fwd_skip_ex.argtypes = [ctypes.POINTER(RenderDesc), vp, vp]
    if lib.gmpi_abi_version() != ABI_VERSION:
        raise GmpiLibraryError(f"ABI mismatch: library {lib.gmpi_abi_version()} != binding {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


def check(rc: int):
    if rc != GMPI_OK:
        raise GmpiLibraryError(f"gmpi error {rc}: {load().gmpi_last_error().decode()}")
