"""ctypes binding of ``csrc/libnr_b200.so`` (the C ABI declared in ``include/nr_b200.h``).

There is no fallback: if the library has not been built the import of any operator
raises, and every call checks that its tensors live on a CUDA device.
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(CSRC, "libnr_b200.so")

ABI_VERSION = 4
NR_OK = 0
NR_ERR_INVALID_ARGUMENT = 1
NR_ERR_CUDA = 2
NR_ERR_WORKSPACE_TOO_SMALL = 3

NR_DRAW_RGB = 1
NR_DRAW_SILHOUETTES = 2
NR_DRAW_DEPTH = 4
NR_DRAW_BACKSIDE = 8
NR_ANTI_ALIASING = 16
NR_DETERMINISTIC = 32
NR_GENERAL_BINNING = 64
NR_SPARSE_MAPS = 128
NR_FINE_TILES = 256
NR_DENSE_RASTER = 512
NR_VIEW_FACES = 1024
NR_FACE_TEXTURES = 2048

# every symbol include/nr_b200.h declares (tests/test_abi.py checks header <-> library <-> this list)
SYMBOLS = (
    "nr_abi_version", "nr_last_error", "nr_num_channels", "nr_event_create", "nr_event_destroy",
    "nr_event_synchronize", "nr_event_query", "nr_deterministic_scratch_bytes", "nr_workspace_bytes", "nr_rasterize_forward", "nr_rasterize_backward",
    "nr_rasterize_backward_lights", "nr_differentiation_backward", "nr_face_index_map_forward_safe", "nr_compute_weight_map",
    "nr_profile_enable", "nr_profile_collect", "nr_camera_partial_blocks", "nr_camera_forward",
    "nr_camera_backward", "nr_camera_exchange_bytes", "nr_camera_backward_shared_allreduce",
)
NR_PROF_SLOTS = 14
PROF_SLOT_NAMES = ("memset", "setup_count", "scan_tiles", "scatter", "sort_long", "raster", "backward",
                   "differentiation_backward", "weight_map_compat", "zbuf_faces", "camera_forward",
                   "camera_backward", "zbuf_resolve", "zbuf_shade")


class RasterConfig(ctypes.Structure):
    """``nrRasterConfig``."""
    _fields_ = [
        ("batch", ctypes.c_int32), ("num_vertices", ctypes.c_int32), ("num_faces", ctypes.c_int32),
        ("image_size", ctypes.c_int32), ("flags", ctypes.c_int32),
        ("near_plane", ctypes.c_float), ("far_plane", ctypes.c_float), ("eps", ctypes.c_float),
        ("depth_min_delta", ctypes.c_float),
        ("num_tex_vertices", ctypes.c_int32), ("tex_height", ctypes.c_int32), ("tex_width", ctypes.c_int32),
    ]


class Lights(ctypes.Structure):
    """``nrLights``."""
    _fields_ = [("num_lights", ctypes.c_int32), ("types", ctypes.c_void_p), ("data", ctypes.c_void_p),
                ("vertex_normals", ctypes.c_void_p), ("grad_vertex_normals", ctypes.c_void_p),
                ("backgrounds", ctypes.c_void_p)]


class ZeroFill(ctypes.Structure):
    """``nrZeroFill``."""
    _fields_ = [("count", ctypes.c_int32), ("ptr", ctypes.c_void_p * 4), ("bytes", ctypes.c_size_t * 4)]


class BinStats(ctypes.Structure):
    """``nrBinStats``."""
    _fields_ = [("total_pairs", ctypes.c_int32), ("max_tile_faces", ctypes.c_int32),
                ("overflow", ctypes.c_int32), ("bad_index", ctypes.c_int32)]


def build(force=False, verbose=False):
    """Compile the CUDA sources for sm_100a with the committed Makefile (nvcc cross-compiles
    without a GPU)."""
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h"))]
    srcs.append(os.path.join(os.path.dirname(_HERE), "include", "nr_b200.h"))
    stale = (not os.path.exists(LIB_PATH) or
             any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs))
    if force or stale:
        cmd = ["make", "-C", CSRC] + (["-B"] if force else [])
        out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if verbose or out.returncode:
            print(out.stdout)
        if out.returncode:
            raise RuntimeError("building libnr_b200.so failed (see output above)")
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "neural_renderer_v2_pytorch_b200: %s is missing. Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` or `make -C %s`. "
            "There is no CPU or PyTorch fallback for this path." % (LIB_PATH, CSRC))
    L = ctypes.CDLL(LIB_PATH)
    vp, i32, i64, f32 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_float
    L.nr_abi_version.restype = ctypes.c_int
    L.nr_abi_version.argtypes = []
    L.nr_last_error.restype = ctypes.c_char_p
    L.nr_last_error.argtypes = []
    L.nr_num_channels.restype = ctypes.c_int
    L.nr_num_channels.argtypes = [i32]
    L.nr_event_create.restype = ctypes.c_int
    L.nr_event_create.argtypes = [ctypes.POINTER(vp)]
    L.nr_event_destroy.restype = ctypes.c_int
    L.nr_event_destroy.argtypes = [vp]
    L.nr_event_synchronize.restype = ctypes.c_int
    L.nr_event_synchronize.argtypes = [vp]
    L.nr_event_query.restype = ctypes.c_int
    L.nr_event_query.argtypes = [vp]
    L.nr_workspace_bytes.restype = ctypes.c_size_t
    L.nr_workspace_bytes.argtypes = [ctypes.POINTER(RasterConfig), i64]
    L.nr_rasterize_forward.restype = ctypes.c_int
    L.nr_rasterize_forward.argtypes = [ctypes.POINTER(RasterConfig), vp, vp, vp, vp, vp, vp, vp, vp, vp,
                                       vp, vp, vp, vp, ctypes.c_size_t, i64, vp, vp, ctypes.POINTER(ZeroFill),
                                       ctypes.POINTER(Lights), vp]
    L.nr_rasterize_backward.restype = ctypes.c_int
    L.nr_rasterize_backward.argtypes = [ctypes.POINTER(RasterConfig)] + [vp] * 14 + [ctypes.POINTER(Lights), vp]
    L.nr_rasterize_backward_lights.restype = ctypes.c_int
    L.nr_rasterize_backward_lights.argtypes = ([ctypes.POINTER(RasterConfig)] + [vp] * 14 +
                                               [ctypes.POINTER(Lights), vp, vp, vp])
    L.nr_deterministic_scratch_bytes.restype = ctypes.c_size_t
    L.nr_deterministic_scratch_bytes.argtypes = [ctypes.POINTER(RasterConfig)]
    L.nr_differentiation_backward.restype = ctypes.c_int
    L.nr_differentiation_backward.argtypes = [vp, vp, vp, i32, i32, i32, vp]
    L.nr_face_index_map_forward_safe.restype = ctypes.c_int
    L.nr_face_index_map_forward_safe.argtypes = [vp, vp, i32, i32, i32, f32, f32, i32, f32, f32, vp]
    L.nr_compute_weight_map.restype = ctypes.c_int
    L.nr_compute_weight_map.argtypes = [vp, vp, vp, i32, i32, i32, vp]
    L.nr_profile_enable.restype = ctypes.c_int
    L.nr_profile_enable.argtypes = [ctypes.c_int]
    L.nr_profile_collect.restype = ctypes.c_int
    L.nr_profile_collect.argtypes = [ctypes.POINTER(ctypes.c_float), ctypes.POINTER(i32)]
    L.nr_camera_partial_blocks.restype = ctypes.c_int
    L.nr_camera_partial_blocks.argtypes = [i32]
    L.nr_camera_forward.restype = ctypes.c_int
    L.nr_camera_forward.argtypes = [vp, vp, vp, vp, i32, i32, i32, f32, i32, vp]
    L.nr_camera_backward.restype = ctypes.c_int
    L.nr_camera_backward.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, f32, i32, vp]
    L.nr_camera_exchange_bytes.restype = ctypes.c_int
    L.nr_camera_exchange_bytes.argtypes = [i32, i32]
    L.nr_camera_backward_shared_allreduce.restype = ctypes.c_int
    L.nr_camera_backward_shared_allreduce.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, f32, i32, i32,
                                                      ctypes.POINTER(vp), vp, vp]
    if L.nr_abi_version() != ABI_VERSION:
        raise RuntimeError("libnr_b200.so ABI version mismatch")
    _lib = L
    return L


def check(rc, what):
    """Turn a non-zero return code into the exception type the reference raises
    (RuntimeError from TORCH_CHECK, ``rasterize_cuda.cpp:5-7``)."""
    if rc != NR_OK:
        msg = lib().nr_last_error().decode("utf-8", "replace")
        raise RuntimeError("%s failed (code %d): %s" % (what, rc, msg))
