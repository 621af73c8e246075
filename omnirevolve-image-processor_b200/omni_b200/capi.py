"""ctypes binding of libomni_b200.so (include/omni_b200.h).  No torch types cross this boundary:
device pointers are plain integers (tensor.data_ptr()), streams are cudaStream_t handles.

There is deliberately no fallback: if the shared library is missing or no CUDA device is present,
importing works but the first call raises."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("OMNI_B200_LIB") or os.path.join(os.path.dirname(_HERE), "lib", "libomni_b200.so")

OMNI_MAX_K = 32
OMNI_MAX_BLUR_K = 31
OMNI_MAX_MORPH_K = 255
ERR_UNSUPPORTED = -3
BITS_LSB_FIRST = 0      # pixel x = bit (x & 7) of byte x >> 3
BITS_MSB_FIRST = 1      # pixel x = bit 7 - (x & 7): the scanline of a 1-bit PNG, numpy.packbits default
PNG_GRAY1 = 0           # packed MSB-first rows -> 1-bit greyscale PNG
PNG_BGR8 = 1            # u8 BGR HWC -> 8-bit RGB PNG
PNG_MAX_SCANLINE = 61440

EXPORTS = [
    "omni_version", "omni_last_error_string", "omni_device_count", "omni_set_fast_path", "omni_ctx_create",
    "omni_ctx_destroy", "omni_host_alloc", "omni_host_free", "omni_resize_area_u8c3", "omni_host_resize_area_u8c3",
    "omni_assign_lab_f32", "omni_assign_rgb_i16wrap", "omni_host_assign_rgb_i16wrap", "omni_layer_masks",
    "omni_edges", "omni_host_edges", "omni_color_edge", "omni_host_color_edge", "omni_count_nonzero",
    "omni_edges_composite", "omni_last_hysteresis_passes", "omni_launch_count", "omni_profile_enable",
    "omni_profile_summary", "omni_thin_zhangsuen", "omni_host_thin_zhangsuen", "omni_swatch_masks", "omni_color_edge_batch", "omni_skeleton_degree",
    "omni_set_table_cache", "omni_host_edges_composite", "omni_color_edge_packed", "omni_host_color_edge_packed",
    "omni_workspace_bytes", "omni_ctx_reserve", "omni_set_assume_binary_masks", "omni_kmeans_lab",
    "omni_thin_zhangsuen_packed", "omni_set_host_bands", "omni_last_band_resends",
    "omni_trace_centerlines", "omni_host_trace_centerlines", "omni_trace_results",
    "omni_kmeans_lab_batch", "omni_color_edge_packed_frames", "omni_host_color_edge_packed_frames",
    "omni_png_bound", "omni_png_encode", "omni_host_png_encode",
]


class EdgeParams(C.Structure):
    """omni_edge_params: 03_edge_detect.py:23-34 knobs."""
    _fields_ = [("morph_k", C.c_int32), ("open_iters", C.c_int32), ("close_iters", C.c_int32),
                ("ksize", C.c_int32), ("low", C.c_double), ("high", C.c_double)]


class OmniError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libomni_b200 error {code}: {msg}")
        self.code = code


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise OmniError(-100, f"{LIB_PATH} not built -- run `python omnirevolve-image-processor_b200/build.py` "
                              "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, sz, i, u8p = C.c_void_p, C.c_size_t, C.c_int, C.c_void_p
    f32p, i64p, epp = C.POINTER(C.c_float), C.POINTER(C.c_int64), C.POINTER(EdgeParams)
    hu8 = C.POINTER(C.c_uint8)
    i32p = C.POINTER(C.c_int32)
    sig = {
        "omni_version": ([], i),
        "omni_last_error_string": ([], C.c_char_p),
        "omni_device_count": ([], i),
        "omni_set_fast_path": ([vp, i], i),
        "omni_set_table_cache": ([vp, i], i),
        "omni_set_host_bands": ([vp, i], i),
        "omni_last_band_resends": ([vp], i),
        "omni_set_assume_binary_masks": ([vp, i], i),
        "omni_workspace_bytes": ([i, i, i, i, i], sz),
        "omni_ctx_reserve": ([vp, i, i, i, i, i], i),
        "omni_kmeans_lab": ([vp, u8p, i, i, sz, i32p, i, i, i, i, C.c_double, C.c_uint64, f32p, C.POINTER(C.c_double), vp], i),
        "omni_kmeans_lab_batch": ([vp, u8p, i, sz, i, i, sz, i32p, i, i, i, i, C.c_double, C.c_uint64, f32p, C.POINTER(C.c_double), vp], i),
        "omni_ctx_create": ([i, C.POINTER(vp)], i),
        "omni_ctx_destroy": ([vp], i),
        "omni_host_alloc": ([sz, C.POINTER(vp)], i),
        "omni_host_free": ([vp], i),
        "omni_resize_area_u8c3": ([vp, u8p, i, i, sz, u8p, i, i, sz, vp], i),
        "omni_host_resize_area_u8c3": ([vp, u8p, i, i, sz, u8p, i, i, sz], i),
        "omni_assign_lab_f32": ([vp, u8p, i, i, sz, f32p, i, hu8, u8p, sz, vp], i),
        "omni_assign_rgb_i16wrap": ([vp, u8p, i, i, sz, hu8, i, u8p, sz, vp], i),
        "omni_host_assign_rgb_i16wrap": ([vp, u8p, i, i, sz, hu8, i, u8p, sz], i),
        "omni_layer_masks": ([vp, u8p, i, i, sz, i, i, i, u8p, sz, sz, vp], i),
        "omni_edges": ([vp, u8p, i, i, i, sz, sz, epp, u8p, sz, sz, vp], i),
        "omni_host_edges": ([vp, u8p, i, i, i, sz, sz, epp, u8p, sz, sz], i),
        "omni_color_edge": ([vp, u8p, i, i, sz, f32p, i, hu8, epp, u8p, sz, u8p, sz, sz, u8p, sz, sz, vp], i),
        "omni_host_color_edge": ([vp, u8p, i, i, sz, f32p, i, hu8, epp, u8p, sz, u8p, sz, sz, u8p, sz, sz, i64p], i),
        "omni_count_nonzero": ([vp, u8p, i, i, i, sz, sz, i64p, vp], i),
        "omni_edges_composite": ([vp, u8p, i, i, i, sz, sz, hu8, u8p, sz, vp], i),
        "omni_host_edges_composite": ([vp, u8p, i, i, i, sz, sz, hu8, u8p, sz], i),
        "omni_last_hysteresis_passes": ([vp], i),
        "omni_launch_count": ([vp], C.c_longlong),
        "omni_profile_enable": ([vp, i], i),
        "omni_profile_summary": ([vp, C.c_char_p, sz], i),
        "omni_thin_zhangsuen": ([vp, u8p, i, i, i, sz, sz, i, u8p, sz, sz, i32p, i32p, vp], i),
        "omni_host_thin_zhangsuen": ([vp, u8p, i, i, i, sz, sz, i, u8p, sz, sz, i32p, i32p], i),
        "omni_thin_zhangsuen_packed": ([vp, u8p, i, i, i, sz, sz, i, i, u8p, sz, sz, i32p, i32p, vp], i),
        "omni_color_edge_batch": ([vp, u8p, i, sz, i, i, sz, f32p, i, hu8, epp, u8p, sz, sz, u8p, sz, sz, vp], i),
        "omni_skeleton_degree": ([vp, u8p, i, i, i, sz, sz, u8p, sz, sz, u8p, sz, sz, vp], i),
        "omni_color_edge_packed": ([vp, u8p, i, sz, i, i, sz, f32p, i, hu8, epp, u8p, sz, sz, u8p, sz, sz, i, i64p, vp], i),
        "omni_host_color_edge_packed": ([vp, u8p, i, sz, i, i, sz, f32p, i, hu8, epp, u8p, sz, sz, u8p, sz, sz, i, i64p], i),
        "omni_color_edge_packed_frames": ([vp, u8p, i, sz, i, i, sz, f32p, i, hu8, epp, u8p, sz, sz, u8p, sz, sz, i, i64p, vp], i),
        "omni_host_color_edge_packed_frames": ([vp, u8p, i, sz, i, i, sz, f32p, i, hu8, epp, u8p, sz, sz, u8p, sz, sz, i, i64p], i),
        "omni_swatch_masks": ([vp, u8p, i, i, sz, i32p, i, i, u8p, sz, sz, i32p, vp], i),
        "omni_trace_centerlines": ([vp, u8p, i, i, i, sz, sz, i64p, vp], i),
        "omni_host_trace_centerlines": ([vp, u8p, i, i, i, sz, sz, i64p], i),
        "omni_trace_results": ([vp, vp, vp, vp], i),
        "omni_png_bound": ([i, i, i], sz),
        "omni_png_encode": ([vp, u8p, i, sz, i, i, sz, i, u8p, sz, i64p, vp], i),
        "omni_host_png_encode": ([vp, u8p, i, sz, i, i, sz, i, u8p, sz, i64p], i),
    }
    for name, (args, res) in sig.items():
        fn = getattr(L, name)
        fn.argtypes, fn.restype = args, res
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise OmniError(rc, lib().omni_last_error_string().decode("utf-8", "replace"))
