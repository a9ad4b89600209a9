"""ctypes binding of libhiccup_b200.so (include/hiccup_b200.h).

There is no CPU fallback: if the library is missing or no CUDA device is usable, the numeric entry
points raise `HicError` / `RuntimeError` rather than computing on the host.
"""
import ctypes
import os
import threading

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HIC_LIB_PATH") or os.path.join(HERE, "libhiccup_b200.so")      # HIC_LIB_PATH: an experimental build (development aid)

c_void_p, c_int, c_int32, c_uint32, c_size_t = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int32,
                                                ctypes.c_uint32, ctypes.c_size_t)
TIE_STATS = 4
TIE_RECORD_BYTES = 16


class HicError(RuntimeError):
    pass


class StreamLayout(ctypes.Structure):
    _fields_ = [("n_images", c_int32), ("skip_first", c_int32), ("blocks_per_image", ctypes.c_int64),
                ("nb", ctypes.c_int64 * 3), ("block_off", ctypes.c_int64 * 3), ("len", ctypes.c_int64 * 3)]


class Geometry(ctypes.Structure):
    _fields_ = [("h", c_int32), ("w", c_int32), ("hc", c_int32), ("wc", c_int32),
                ("nby_l", c_int32), ("nbx_l", c_int32), ("nby_c", c_int32), ("nbx_c", c_int32),
                ("nb_l", ctypes.c_int64), ("nb_c", ctypes.c_int64), ("blocks_per_image", ctypes.c_int64),
                ("out_h", c_int32), ("out_w", c_int32)]


class HicfileEnv(ctypes.Structure):
    _fields_ = [("np_pre", c_void_p), ("np_mid", c_void_p), ("head", c_void_p),
                ("np_pre_len", c_uint32), ("np_mid_len", c_uint32), ("head_len", c_uint32), ("reserved", c_uint32)]


class HicfileBatch(ctypes.Structure):
    _fields_ = [("n_files", ctypes.c_uint64), ("tables_per_file", c_uint32), ("n_trail", c_uint32),
                ("stream_of", c_void_p), ("flag_mode", c_void_p), ("index", c_void_p), ("symbols", c_void_p), ("packed", c_void_p),
                ("data", c_void_p), ("byte_off", c_void_p), ("byte_len", c_void_p), ("lead", c_void_p), ("lead_len", ctypes.c_uint64),
                ("trail", c_void_p), ("trail_len", c_void_p)]


class BandCarry(ctypes.Structure):
    _fields_ = [("carry_zeros", c_int32), ("prev_dc", c_int32), ("more_after", c_int32), ("closes_stream", c_int32)]


class WaveletGeometry(ctypes.Structure):
    _fields_ = [("h", c_int32), ("w", c_int32), ("lh", c_int32 * 4), ("lw", c_int32 * 4),
                ("band_off", ctypes.c_int64 * 10), ("len", ctypes.c_int64)]


class WaveletPyramid(ctypes.Structure):
    _fields_ = [("h", c_int32), ("w", c_int32), ("levels", c_int32), ("n_bands", c_int32), ("lh", c_int32 * 6),
                ("lw", c_int32 * 6), ("band_off", ctypes.c_int64 * 16), ("len", ctypes.c_int64)]


class WaveletParams(ctypes.Structure):
    _fields_ = [("levels", c_int32), ("reserved", c_int32), ("multiplier", ctypes.c_double),
                ("threshold", ctypes.c_double), ("threshold_index", ctypes.c_int64)]


#: every symbol include/hiccup_b200.h declares -> (restype, argtypes)
SIGNATURES = {
    "hic_version": (c_int, []),
    "hic_last_error": (ctypes.c_char_p, []),
    "hic_device_count": (c_int, [ctypes.POINTER(c_int)]),
    "hic_set_device": (c_int, [c_int]),
    "hic_get_device": (c_int, [ctypes.POINTER(c_int)]),
    "hic_device_name": (c_int, [ctypes.c_char_p, c_size_t]),
    "hic_malloc": (c_int, [ctypes.POINTER(c_void_p), c_size_t]),
    "hic_free": (c_int, [c_void_p]),
    "hic_host_alloc": (c_int, [ctypes.POINTER(c_void_p), c_size_t]),
    "hic_host_free": (c_int, [c_void_p]),
    "hic_host_register": (c_int, [c_void_p, c_size_t]),
    "hic_host_unregister": (c_int, [c_void_p]),
    "hic_ticket_take": (c_int, [c_void_p, ctypes.c_int64, ctypes.POINTER(ctypes.c_int64)]),
    "hic_memcpy_h2d": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
    "hic_memcpy_d2h": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
    "hic_memset": (c_int, [c_void_p, c_int, c_size_t, c_void_p]),
    "hic_stream_create": (c_int, [ctypes.POINTER(c_void_p)]),
    "hic_stream_destroy": (c_int, [c_void_p]),
    "hic_stream_sync": (c_int, [c_void_p]),
    "hic_set_blocking_sync": (c_int, [c_int]),
    "hic_profile_enable": (c_int, [c_int]),
    "hic_profile_report": (c_int, [ctypes.c_char_p, c_size_t]),
    "hic_profile_timeline": (c_int, [ctypes.c_char_p, c_size_t]),
    "hic_dct_geometry_of": (c_int, [c_int32, c_int32, ctypes.POINTER(Geometry)]),
    "hic_dct_tie_capacity": (c_int, [c_int32, c_int32, c_int32, ctypes.POINTER(c_uint32)]),
    "hic_dct_forward": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_uint32, c_void_p, c_void_p]),
    "hic_blocks_to_planes": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hic_planes_to_blocks": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "hic_dct_inverse": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p,
                                c_void_p, c_uint32, c_void_p, c_void_p]),
    "hic_wavelet_geometry_of": (c_int, [c_int32, c_int32, ctypes.POINTER(WaveletGeometry)]),
    "hic_wavelet_forward": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "hic_wavelet_inverse": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "hic_wavelet_flat_to_bands": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "hic_wavelet_bands_to_flat": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "hic_wavelet_pyramid_of": (c_int, [c_int32, c_int32, c_int32, ctypes.POINTER(WaveletPyramid)]),
    "hic_wavelet_general_work_bytes": (c_int, [c_int32, c_int32, c_int32, ctypes.POINTER(c_size_t)]),
    "hic_wavelet_forward_general": (c_int, [c_void_p, c_int32, c_int32, c_int32, ctypes.POINTER(WaveletParams), c_void_p, c_void_p, c_void_p]),
    "hic_wavelet_inverse_general": (c_int, [c_void_p, c_int32, c_int32, c_int32, ctypes.POINTER(WaveletParams), c_void_p, c_void_p, c_void_p]),
    "hic_wavelet_scaled_general": (c_int, [c_void_p, c_int32, c_int32, c_int32, ctypes.POINTER(WaveletParams), c_int32, c_void_p,
                                           c_void_p, c_void_p]),
    "hic_wavelet_region": (c_int, [c_void_p, c_int32, c_int32, c_int32, ctypes.POINTER(WaveletParams), c_int32, c_void_p, c_int32,
                                   c_int32, c_void_p, c_size_t, c_void_p, c_void_p]),
    "hic_wavelet_flat_to_bands_general": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "hic_wavelet_bands_to_flat_general": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "hic_layout_dct": (c_int, [c_int32, c_int32, c_int32, ctypes.POINTER(StreamLayout)]),
    "hic_layout_flat": (c_int, [c_int32, ctypes.c_int64, ctypes.POINTER(StreamLayout)]),
    "hic_entropy_plan_create": (c_int, [ctypes.POINTER(StreamLayout), c_int32, ctypes.POINTER(c_void_p)]),
    "hic_entropy_plan_destroy": (c_int, [c_void_p]),
    "hic_entropy_symbolize": (c_int, [c_void_p, c_void_p, c_void_p]),
    "hic_entropy_scan": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hic_entropy_emit": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "hic_entropy_histograms": (c_int, [c_void_p, c_void_p, c_void_p, ctypes.c_uint64, ctypes.POINTER(ctypes.c_uint64),
                                       c_void_p, c_void_p]),
    "hic_entropy_set_codes": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, ctypes.c_uint64, c_void_p, c_void_p,
                                      c_void_p, c_void_p]),
    "hic_entropy_build_codes": (c_int, [c_void_p, c_void_p]),
    "hic_entropy_build_codes_device": (c_int, [c_void_p, c_void_p]),
    "hic_entropy_device_tables": (c_int, [c_void_p, ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p),
                                          ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p)]),
    "hic_decode_set_tables_device": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, ctypes.c_uint64, c_void_p]),
    "hic_entropy_stream_info": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                        ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64)]),
    "hic_entropy_tables": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "hic_entropy_tables_packed": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hic_entropy_pack": (c_int, [c_void_p, c_void_p, c_void_p]),
    "hic_huffman_build_host": (c_int, [c_void_p, c_uint32, c_void_p, c_void_p]),
    "hic_entropy_symbol_buffers": (c_int, [c_void_p, ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p),
                                           ctypes.POINTER(c_void_p)]),
    "hic_decode_plan_create": (c_int, [ctypes.POINTER(StreamLayout), ctypes.POINTER(c_void_p)]),
    "hic_decode_plan_destroy": (c_int, [c_void_p]),
    "hic_decode_set_tables": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hic_decode_set_tables_packed": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, ctypes.c_uint64, c_void_p]),
    "hic_decode_run": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hic_hicfile_pack_rows": (c_int, [c_void_p, c_void_p, c_void_p, ctypes.c_uint64, c_void_p, c_void_p, c_uint32, c_void_p, c_uint32,
                                      c_void_p, ctypes.c_uint64, c_void_p]),
    "hic_hicfile_pack_table": (c_int, [c_void_p, c_void_p, c_void_p, ctypes.c_uint64, c_void_p, c_void_p, c_uint32, c_void_p, c_uint32,
                                       c_void_p, c_uint32, c_void_p, ctypes.c_uint64, c_void_p]),
    "hic_hicfile_parse_table": (c_int, [c_void_p, ctypes.c_uint64, c_void_p, c_uint32, c_void_p, c_uint32, c_void_p, c_void_p, c_void_p,
                                        c_void_p, ctypes.c_uint64, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_int32)]),
    "hic_hicfile_files_bound": (c_int, [ctypes.POINTER(HicfileEnv), ctypes.POINTER(HicfileBatch), c_void_p, c_uint32]),
    "hic_hicfile_pack_files": (c_int, [ctypes.POINTER(HicfileEnv), ctypes.POINTER(HicfileBatch), c_void_p, c_void_p, c_void_p, c_uint32]),
    "hic_hicfile_scan_files": (c_int, [c_void_p, c_void_p, ctypes.c_uint64, c_uint32, c_uint32, c_void_p, c_void_p, c_void_p, c_void_p, c_uint32]),
    "hic_hicfile_parse_files": (c_int, [ctypes.POINTER(HicfileEnv), c_void_p, ctypes.c_uint64, c_uint32, c_uint32, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_uint32]),
    "hic_hicfile_parse_rows": (c_int, [c_void_p, c_void_p, ctypes.c_uint64, c_void_p, c_uint32, c_void_p, c_uint32, c_void_p, c_void_p,
                                       c_void_p, c_void_p, ctypes.POINTER(ctypes.c_int64)]),
    "hic_decode_set_data_bytes": (c_int, [c_void_p, ctypes.c_uint64]),
    "hic_decode_sync": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, ctypes.POINTER(ctypes.c_uint64), c_void_p]),
    "hic_decode_export_restarts": (c_int, [c_void_p, c_void_p, c_void_p, ctypes.c_uint64, c_void_p]),
    "hic_decode_run_restarts": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, ctypes.c_uint64, c_void_p, c_void_p]),
    "hic_decode_run_dc": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, ctypes.c_uint64, c_void_p, c_void_p]),
    "hic_dct_thumbnail_shape": (c_int, [c_int32, c_int32, ctypes.POINTER(c_int32), ctypes.POINTER(c_int32)]),
    "hic_dct_thumbnail": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "hic_dct_region_blocks": (c_int, [c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, ctypes.POINTER(c_int32)]),
    "hic_dct_region_sizes": (c_int, [c_int32, c_int32, c_int32, c_int32, c_int32, ctypes.POINTER(c_size_t), ctypes.POINTER(c_uint32)]),
    "hic_dct_region": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int32, c_int32, c_void_p, c_size_t, c_void_p,
                               c_uint32, c_void_p, c_void_p, c_void_p]),
    "hic_dct_scaled_shape": (c_int, [c_int32, c_int32, c_int32, ctypes.POINTER(c_int32), ctypes.POINTER(c_int32)]),
    "hic_dct_scaled_sizes": (c_int, [c_int32, c_int32, c_int32, c_int32, ctypes.POINTER(c_size_t), ctypes.POINTER(c_uint32)]),
    "hic_dct_scaled": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_size_t, c_void_p, c_uint32, c_void_p,
                               c_void_p, c_void_p]),
    "hic_dct_scaled_region_blocks": (c_int, [c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, ctypes.POINTER(c_int32)]),
    "hic_dct_scaled_region_sizes": (c_int, [c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, ctypes.POINTER(c_size_t),
                                            ctypes.POINTER(c_uint32)]),
    "hic_dct_scaled_region": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int32, c_int32, c_void_p, c_size_t,
                                      c_void_p, c_uint32, c_void_p, c_void_p, c_void_p]),
    "hic_dct_thumbnail_region": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int32, c_int32, c_void_p, c_size_t,
                                         c_void_p, c_void_p]),
}

_lock = threading.Lock()
_lib = None


def load():
    """Load the shared library and bind every declared symbol (no CUDA call is made)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise HicError("libhiccup_b200.so is not built (%s); run `python -m hiccup_b200.build` -- "
                           "there is no CPU fallback" % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(lib, name)       # AttributeError if the header and the library diverge
            fn.restype, fn.argtypes = restype, argtypes
        _lib = lib
        return lib


def check(rc):
    if rc != 0:
        msg = load().hic_last_error()
        raise HicError("hiccup_b200 error %d: %s" % (rc, (msg or b"").decode("utf-8", "replace")))


_device_ready = False


def require_device():
    """Fail loudly when there is no CUDA device (the product has no host path)."""
    global _device_ready
    if _device_ready:
        return
    lib = load()
    n = c_int(0)
    rc = lib.hic_device_count(ctypes.byref(n))
    if rc != 0 or n.value < 1:
        raise HicError("no CUDA device is available; hiccup_b200 has no CPU fallback (%s)"
                       % (lib.hic_last_error() or b"").decode("utf-8", "replace"))
    _device_ready = True


def geometry(h, w):
    g = Geometry()
    check(load().hic_dct_geometry_of(int(h), int(w), ctypes.byref(g)))
    return g


def thumbnail_shape(h, w):
    """(th, tw) of the 1/8-scale thumbnail of a DCT-mode image of h x w (host only)."""
    th, tw = c_int32(), c_int32()
    check(load().hic_dct_thumbnail_shape(int(h), int(w), ctypes.byref(th), ctypes.byref(tw)))
    return int(th.value), int(tw.value)


def region_blocks(h, w, top, left, rh, rw):
    """The block rectangles a window of rh x rw at (top, left) of the decoded image selects (host only):
    ((by, bx, nby, nbx) of the luminance plane, the same of each chroma plane).  HicError for an invalid window."""
    rect = (c_int32 * 8)()
    check(load().hic_dct_region_blocks(int(h), int(w), int(top), int(left), int(rh), int(rw), rect))
    return tuple(rect[0:4]), tuple(rect[4:8])


def region_sizes(n, h, w, rh, rw):
    """(work bytes, tie capacity) hic_dct_region needs for n windows of rh x rw (host only)."""
    work, cap = c_size_t(), c_uint32()
    check(load().hic_dct_region_sizes(int(n), int(h), int(w), int(rh), int(rw), ctypes.byref(work), ctypes.byref(cap)))
    return int(work.value), int(cap.value)


def region_origins(h, w, origins, size, scale=1):
    """Check windows of size = (rh, rw) at origins ((n, 2) (top, left)) against the h x w image's decoded output
    (out_h x out_w), or with scale 2, 4 or 8 against its 1/scale image (ceil(out_h / scale) x ceil(out_w / scale)), on
    the host: the origins as a contiguous (n, 2) int32 array, or ValueError."""
    g = geometry(h, w)
    scale = region_scale_arg(scale)
    ih, iw = (g.out_h, g.out_w) if scale == 1 else (-(-g.out_h // scale), -(-g.out_w // scale))
    return _window_origins(ih, iw, "decoded image" if scale == 1 else "1/%d-scale image" % scale, origins, size)


def wavelet_region_origins(h, w, levels, origins, size, scale=1):
    """region_origins() for a wavelet file of `levels` levels and h x w (multiples of 2^levels): windows of the
    full-resolution image (scale 1) or of the (h / scale) x (w / scale) image, scale = 2^k with 1 <= k <= levels."""
    levels = int(levels)
    k = wavelet_scale_arg(scale, levels, lowest=0)
    if h % (1 << levels) or w % (1 << levels):
        raise ValueError("a region decode of %d levels needs sides that are multiples of %d (got %dx%d)" % (levels, 1 << levels, h, w))
    return _window_origins(h >> k, w >> k, "image" if k == 0 else "1/%d-scale image" % (1 << k), origins, size)


def _window_origins(ih, iw, what, origins, size):
    """The origins ((n, 2) of (top, left)) of windows of size = (rh, rw) inside an ih x iw image (`what`, for the
    message) as a contiguous (n, 2) int32 array, or ValueError."""
    rh, rw = (int(v) for v in size)
    o = np.asarray(origins)
    if o.ndim != 2 or o.shape[1] != 2 or o.shape[0] < 1 or not np.issubdtype(o.dtype, np.integer):
        raise ValueError("origins must be a non-empty (n, 2) integer array of (top, left), got shape %r" % (o.shape,))
    o = o.astype(np.int64)
    if rh < 1 or rw < 1:
        raise ValueError("empty region %dx%d" % (rh, rw))
    bad = (o[:, 0] < 0) | (o[:, 1] < 0) | (o[:, 0] + rh > ih) | (o[:, 1] + rw > iw)
    if bad.any():
        i = int(np.argmax(bad))
        raise ValueError("region %dx%d at (%d, %d) is not inside the %dx%d %s" % (rh, rw, o[i, 0], o[i, 1], ih, iw, what))
    return np.ascontiguousarray(o, np.int32)


def region_scale_arg(scale):
    """scale as an int if it is a region decode's scale -- 1 (full resolution), 2, 4 or 8 -- else ValueError."""
    if isinstance(scale, bool) or not isinstance(scale, (int, np.integer)) or int(scale) not in (1, 2, 4, 8):
        raise ValueError("a region's scale must be 1, 2, 4 or 8 (got %r)" % (scale,))
    return int(scale)


def scaled_region_blocks(h, w, scale, top, left, rh, rw):
    """region_blocks() for a window of the 1/scale image, scale 2 or 4 (host only)."""
    rect = (c_int32 * 8)()
    check(load().hic_dct_scaled_region_blocks(int(h), int(w), int(scale), int(top), int(left), int(rh), int(rw), rect))
    return tuple(rect[0:4]), tuple(rect[4:8])


def scaled_region_sizes(n, h, w, scale, rh, rw):
    """(work bytes, tie capacity) hic_dct_scaled_region (scale 2, 4) or hic_dct_thumbnail_region (scale 8) needs for n
    windows of rh x rw of the 1/scale image (host only)."""
    work, cap = c_size_t(), c_uint32()
    check(load().hic_dct_scaled_region_sizes(int(n), int(h), int(w), int(scale), int(rh), int(rw), ctypes.byref(work),
                                             ctypes.byref(cap)))
    return int(work.value), int(cap.value)


def scale_arg(scale):
    """scale as an int if it is 2 or 4 (the scaled decode's factors; 8 is the thumbnail), else ValueError."""
    if isinstance(scale, bool) or not isinstance(scale, (int, np.integer)) or int(scale) not in (2, 4):
        raise ValueError("scale must be 2 or 4 (got %r; 1/8 scale is the thumbnail)" % (scale,))
    return int(scale)


def scaled_shape(h, w, scale):
    """(sh, sw) = (ceil(out_h / scale), ceil(out_w / scale)) of the scaled decode (host only)."""
    sh, sw = c_int32(), c_int32()
    check(load().hic_dct_scaled_shape(int(h), int(w), int(scale), ctypes.byref(sh), ctypes.byref(sw)))
    return int(sh.value), int(sw.value)


def scaled_sizes(n, h, w, scale):
    """(work bytes, tie capacity) hic_dct_scaled needs for n images (host only)."""
    work, cap = c_size_t(), c_uint32()
    check(load().hic_dct_scaled_sizes(int(n), int(h), int(w), int(scale), ctypes.byref(work), ctypes.byref(cap)))
    return int(work.value), int(cap.value)


def tie_capacity(n, h, w):
    """Records the tie buffer of hic_dct_forward must hold (one per block + K1's flag words)."""
    cap = c_uint32()
    check(load().hic_dct_tie_capacity(int(n), int(h), int(w), ctypes.byref(cap)))
    return int(cap.value)


def current_device():
    d = c_int()
    check(load().hic_get_device(ctypes.byref(d)))
    return int(d.value)


class _BufferPool:
    """Freed device buffers of the single-image entry points, kept for the next call: compression.* and codec.*
    allocate some twenty scratch buffers per image, and cudaMalloc / cudaFree serialise on a driver lock (tens of
    milliseconds per call when anything else -- an nvidia-smi poll, another thread -- holds it).  Exact-size
    reuse, per device, bounded; buffers above MAX_ONE bytes are never kept."""
    MAX_ONE = 64 << 20
    MAX_TOTAL = 512 << 20

    def __init__(self):
        self.lock = threading.Lock()
        self.free = {}            # (device, nbytes) -> [ptr, ...]
        self.total = 0
        self.enabled = os.environ.get("HIC_NO_POOL") is None

    def take(self, nbytes):
        if not self.enabled or nbytes > self.MAX_ONE:
            return None
        key = (current_device(), nbytes)
        with self.lock:
            ptrs = self.free.get(key)
            if ptrs:
                self.total -= nbytes
                return ptrs.pop()
        return None

    def give(self, ptr, nbytes):
        if not self.enabled or nbytes > self.MAX_ONE:
            return False
        key = (current_device(), nbytes)
        with self.lock:
            if self.total + nbytes > self.MAX_TOTAL:
                return False
            self.free.setdefault(key, []).append(ptr)
            self.total += nbytes
        return True

    def clear(self):
        """Return everything to the driver (buffers of other devices are freed on their own device)."""
        with self.lock:
            items, self.free, self.total = list(self.free.items()), {}, 0
        lib = load()
        here = current_device() if items else 0
        for (dev, _), ptrs in items:
            lib.hic_set_device(dev)
            for p in ptrs:
                lib.hic_free(p)
        if items:
            lib.hic_set_device(here)


POOL = _BufferPool()


class DeviceBuffer:
    """A device allocation owned through the C ABI (no torch involved).  pooled=True: taken from / returned to
    POOL (the single-image entry points); the batch codecs own their buffers for their whole life."""

    def __init__(self, nbytes, pooled=False):
        require_device()
        self.nbytes = int(nbytes)
        self.pooled = pooled
        ptr = POOL.take(self.nbytes) if pooled else None
        if ptr is None:
            p = c_void_p()
            check(load().hic_malloc(ctypes.byref(p), self.nbytes))
            ptr = p.value
        self.ptr = ptr

    def upload(self, array, stream=None):
        a = np.ascontiguousarray(array)
        assert a.nbytes <= self.nbytes
        check(load().hic_memcpy_h2d(self.ptr, a.ctypes.data, a.nbytes, stream))
        return a            # keep alive until the stream is synchronised

    def download(self, dtype, count, stream=None, offset=0, out=None):
        """Device -> host.  `out`: a preallocated (ideally pinned) array to fill instead of a new one."""
        out = np.empty(int(count), dtype=dtype) if out is None else out
        assert out.dtype == np.dtype(dtype) and out.size == int(count) and out.flags.c_contiguous
        assert offset + out.nbytes <= self.nbytes
        check(load().hic_memcpy_d2h(out.ctypes.data, self.ptr + offset, out.nbytes, stream))
        check(load().hic_stream_sync(stream))
        return out

    def zero(self, stream=None):
        check(load().hic_memset(self.ptr, 0, self.nbytes, stream))

    def free(self):
        if self.ptr:
            if not (self.pooled and POOL.give(self.ptr, self.nbytes)):
                load().hic_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def scratch(nbytes):
    """A pooled device buffer for the single-image entry points (see _BufferPool)."""
    return DeviceBuffer(nbytes, pooled=True)


class PinnedBuffer:
    """Page-locked host memory owned through the C ABI; `array(dtype, count)` views it as numpy."""

    def __init__(self, nbytes):
        require_device()
        self.nbytes = int(nbytes)
        p = c_void_p()
        check(load().hic_host_alloc(ctypes.byref(p), max(self.nbytes, 1)))
        self.ptr = p.value
        self._raw = (ctypes.c_uint8 * max(self.nbytes, 1)).from_address(self.ptr)

    def array(self, dtype=np.uint8, count=None, offset=0):
        item = np.dtype(dtype).itemsize
        count = (self.nbytes - offset) // item if count is None else int(count)
        assert offset + count * item <= self.nbytes
        return np.frombuffer(self._raw, dtype=dtype, count=count, offset=offset)

    def free(self):
        if self.ptr:
            self._raw = None
            load().hic_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def wavelet_geometry(h, w):
    g = WaveletGeometry()
    check(load().hic_wavelet_geometry_of(int(h), int(w), ctypes.byref(g)))
    return g


def wavelet_pyramid(h, w, levels):
    g = WaveletPyramid()
    check(load().hic_wavelet_pyramid_of(int(h), int(w), int(levels), ctypes.byref(g)))
    return g


def wavelet_scale_arg(scale, levels, lowest=1):
    """k for a wavelet scaled decode's scale = 2^k of a file of `levels` levels (lowest <= k <= levels; a region decode
    takes lowest = 0, the full-resolution image), else ValueError."""
    levels = int(levels)
    if isinstance(scale, bool) or not isinstance(scale, (int, np.integer)) or int(scale) < 1 << lowest \
            or int(scale) & (int(scale) - 1) or int(scale) > 1 << levels:
        raise ValueError("scale must be 2^k with %d <= k <= %d, the file's levels (got %r)" % (lowest, levels, scale))
    return int(scale).bit_length() - 1


def wavelet_work_bytes(n, h, w):
    out = c_size_t()
    check(load().hic_wavelet_general_work_bytes(int(n), int(h), int(w), ctypes.byref(out)))
    return int(out.value)


def layout_dct(n, h, w):
    lay = StreamLayout()
    check(load().hic_layout_dct(int(n), int(h), int(w), ctypes.byref(lay)))
    return lay


def layout_flat(n, length):
    lay = StreamLayout()
    check(load().hic_layout_flat(int(n), int(length), ctypes.byref(lay)))
    return lay


def profile_enable(on=True):
    check(load().hic_profile_enable(1 if on else 0))


def profile_report():
    """{"kernel name": (total_ms, launches)} since the last report."""
    import json
    buf = ctypes.create_string_buffer(1 << 16)
    check(load().hic_profile_report(buf, len(buf)))
    return {k: (v[0], v[1]) for k, v in json.loads(buf.value.decode()).items()}


def profile_timeline():
    """[(kernel, stream number, start ms, end ms)] of the spans recorded since the last report."""
    import json
    buf = ctypes.create_string_buffer(1 << 24)
    check(load().hic_profile_timeline(buf, len(buf)))
    return [tuple(e) for e in json.loads(buf.value.decode())]


def stream_create():
    """A new non-blocking CUDA stream (as the integer handle the C ABI takes)."""
    require_device()
    st = c_void_p()
    check(load().hic_stream_create(ctypes.byref(st)))
    return st.value


def stream_destroy(stream):
    if stream:
        load().hic_stream_destroy(stream)


def sync(stream=None):
    check(load().hic_stream_sync(stream))
