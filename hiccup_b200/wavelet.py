"""Wavelet ("HIC") mode, drop-in for the reference's four wavelet entry points.

    wavelet_compression(rgb)      compression.py:59-85      wavelet_encode(c)    codec.py:116-163
    wavelet_decompression(c)      compression.py:88-100     wavelet_decode(hic)  codec.py:199-239
    wavelet_scaled(hic, scale)    no reference counterpart: the 1/2- to 1/2^L-scale image (include/hiccup_b200.h)
    wavelet_region(hic, top, left, height, width, scale)    no reference counterpart: one window of the full or 1/scale image

The numeric work runs in csrc/hic_wavelet.cu (K9 / K10, the fused kernels for the default settings),
csrc/hic_wavelet_general.cu (any WAVELET_NUM_LEVELS in 1..5, multiplier, threshold and quality factor:
settings.py:12-16) and the shared entropy kernels in flat mode (include/hiccup_b200.h).  The transform
restates PyWavelets' db1 wavedec2 / waverec2 in float64; PyWavelets itself could not be installed, so
coefficient values are parity-checked against the reference run on oracle/pywt_standin.py only
(DESIGN.md section 8).
"""
import ctypes

import numpy as np

from hiccup_b200 import _lib, entropy, hicimage, iohelper, model, settings

CHANNELS = ("lum", "cr", "cb")


def band_shapes(g):
    """Shapes of the 3 L + 1 sub-bands [cA_L, cH_L, cV_L, cD_L, cH_(L-1), ..., cD_1] of one channel."""
    levels = int(getattr(g, "levels", 3))
    lvl = [levels] + [l for l in range(levels, 0, -1) for _ in range(3)]
    return [(int(g.lh[l]), int(g.lw[l])) for l in lvl]


def _params(g):
    """settings -> hic_wavelet_params for a channel of g.len coefficients (quantization.py:84-94 for the index)."""
    p = _lib.WaveletParams()
    p.levels = int(settings.WAVELET_NUM_LEVELS)
    p.multiplier = float(settings.WAVELET_SUBBAND_QUANTIZATION_MULTIPLIER)
    p.threshold = float(settings.WAVELET_THRESHOLD)
    p.threshold_index = -1
    if settings.WAVELET_QUALITY_FACTOR != 1:
        n = int(g.len)
        keep = int(np.ceil(n * settings.WAVELET_QUALITY_FACTOR))
        if keep < 1:
            raise IndexError("list index out of range")          # what the reference's s[len(vals)] raises
        p.threshold_index = n - keep
    return p


def _as_rgb(rgb):
    a = np.asarray(rgb)
    if a.ndim != 3 or a.shape[2] != 3:
        raise ValueError("expected an H x W x 3 image, got shape %r" % (a.shape,))
    if a.dtype != np.uint8:
        raise TypeError("expected uint8 pixels, got %s" % a.dtype)
    return np.ascontiguousarray(a)


def _flat_elems(g):
    return 64 * ((int(g.len) + 63) // 64)


def forward_device(d_rgb, n, h, w, stream=None):
    """K9 (default settings) or the general path on a device-resident batch -> (flat stream buffer, geometry)."""
    lib = _lib.load()
    if settings.wavelet_defaults():
        g = _lib.wavelet_geometry(h, w)
        flat = _lib.scratch(2 * _flat_elems(g) * 3 * n)
        _lib.check(lib.hic_wavelet_forward(d_rgb, n, h, w, flat.ptr, stream))
        return flat, g
    g = _lib.wavelet_pyramid(h, w, settings.WAVELET_NUM_LEVELS)
    flat = _lib.scratch(2 * _flat_elems(g) * 3 * n)
    work = _lib.scratch(_lib.wavelet_work_bytes(n, h, w))
    try:
        params = _params(g)
        _lib.check(lib.hic_wavelet_forward_general(d_rgb, n, h, w, ctypes.byref(params), work.ptr, flat.ptr, stream))
        _lib.sync(stream)
    finally:
        work.free()
    return flat, g


def _split_bands(arr, g, dtype):
    """(3, len) concatenated raster bands -> {channel: [10 arrays]}."""
    shapes = band_shapes(g)
    out = {}
    for ci, ch in enumerate(CHANNELS):
        bands, off = [], 0
        for (bh, bw) in shapes:
            bands.append(np.ascontiguousarray(arr[ci, off:off + bh * bw].reshape(bh, bw)).astype(dtype))
            off += bh * bw
        out[ch] = bands
    return out


def wavelet_compression(rgb_image: np.ndarray) -> model.CompressedImage:
    """RGB -> YCrCb, x - 256, L-level db1, sub-band quantisation, thresholds; 3 L + 1 int32 sub-bands per channel."""
    settings.check_wavelet_supported()
    _lib.require_device()
    lib = _lib.load()
    img = _as_rgb(rgb_image)
    h, w = img.shape[:2]
    d_rgb = _lib.scratch(img.nbytes)
    d_rgb.upload(img)
    flat, g = forward_device(d_rgb.ptr, 1, h, w)
    d_bands = _lib.scratch(4 * int(g.len) * 3)
    _lib.check(lib.hic_wavelet_flat_to_bands_general(flat.ptr, 1, h, w, _levels_of(g), d_bands.ptr, None))
    arr = d_bands.download(np.int32, int(g.len) * 3).reshape(3, int(g.len))
    for b in (d_rgb, flat, d_bands):
        b.free()
    return model.CompressedImage.from_dict(_split_bands(arr, g, np.int32))


def _levels_of(g):
    return int(getattr(g, "levels", 3))


def _image_shape_of(bands):
    """(h1, w1, levels) of a channel's sub-band list: the level-1 bands are ceil(n / 2) on a side."""
    if len(bands) < 4 or (len(bands) - 1) % 3 or (len(bands) - 1) // 3 > 5:
        raise ValueError("expected 3 L + 1 sub-bands per channel (L in 1..5), got %d" % len(bands))
    h1, w1 = (int(v) for v in np.asarray(bands[-1]).shape)
    return h1, w1, (len(bands) - 1) // 3


def _bands_to_device_flat(compressed, stream=None):
    """Upload a wavelet CompressedImage and build the flat zigzag stream on the device."""
    lib = _lib.load()
    d = compressed.as_dict
    h1, w1, levels = _image_shape_of(d["lum"])
    # the image shape is not stored: any (h, w) with ceil(h/2) = h1 gives the same sub-band shapes
    h, w = 2 * h1, 2 * w1
    g = _lib.wavelet_pyramid(h, w, levels)
    shapes = band_shapes(g)
    cat = np.empty((3, int(g.len)), np.int32)
    max_abs = 0
    for ci, ch in enumerate(CHANNELS):
        bands = d[ch]
        if len(bands) != len(shapes):
            raise ValueError("expected %d sub-bands in channel %s" % (len(shapes), ch))
        off = 0
        for b, shp in zip(bands, shapes):
            a = np.asarray(b)
            if a.shape != shp:
                raise ValueError("sub-band shape %r does not fit a %d-level db1 pyramid (expected %r)" % (a.shape, levels, shp))
            if a.dtype.kind == "f":
                r = np.rint(a)
                if not np.array_equal(r, a):
                    raise NotImplementedError("non-integral coefficients are not on the CUDA entropy path")
                a = r
            a = a.astype(np.int64)
            if a.size:
                max_abs = max(max_abs, int(np.abs(a).max()))
            cat[ci, off:off + a.size] = a.reshape(-1)
            off += a.size
    if max_abs > 32767:
        raise ValueError("coefficients up to %d do not fit the int16 symbol path" % max_abs)
    d_bands = _lib.scratch(cat.nbytes)
    d_bands.upload(cat, stream)
    flat = _lib.scratch(2 * _flat_elems(g) * 3)
    _lib.check(lib.hic_wavelet_bands_to_flat_general(d_bands.ptr, 1, h, w, levels, flat.ptr, stream))
    _lib.sync(stream)
    d_bands.free()
    return flat, g, max_abs


def _value_bins(max_abs):
    bins = entropy.DEFAULT_VALUE_BINS
    while bins // 2 < max_abs + 1:
        bins *= 2
    return bins


def _wavelet_symbol(v):
    """Types the reference's run-length symbols have when pickled (SURVEY hard part 3): non-zero values
    are the sub-band's np.int32 scalars (transform.zigzag, transform.py:134), zero comes from the Python
    literals of codec.run_length_coding (codec.py:65,89)."""
    return 0 if v == 0 else np.int32(v)


def encode_streams_to_hic(res, g, image=0):
    """EncodedStreams of a flat-mode batch -> the reference's HicImage for one image (14 payloads:
    3 value tables, 3 length tables, 3 value bit strings, 3 length bit strings, cA3 shape, cD1 shape;
    codec.py:147-163)."""
    tables, bits = [], []
    for kind in (entropy.KIND_VALUE, entropy.KIND_LENGTH):
        for c in range(3):
            s = (image * 3 + c) * 3 + kind
            sym, lens, codes = res.stream_rows(s)
            # (_wavelet_symbol: non-zero values are np.int32 scalars in the pickles, zero and the zero counts Python ints)
            flags = (np.asarray(sym) != 0).astype(np.uint8) if kind == entropy.KIND_VALUE else False
            tables.append(hicimage.PayloadStringP.from_arrays(sym, lens, codes, flags))
            bits.append(hicimage.BitStringP.from_framed(res.framed(s)))
    shapes = band_shapes(g)
    payloads = tables + bits + [hicimage.TupP(*shapes[0]), hicimage.TupP(*shapes[-1])]
    return hicimage.HicImage.wavelet_image(payloads)


def wavelet_encode(compressed: model.CompressedImage) -> hicimage.HicImage:
    settings.check_wavelet_supported()
    _lib.require_device()
    flat, g, max_abs = _bands_to_device_flat(compressed)
    layout = _lib.layout_flat(1, int(g.len))
    enc = entropy.cached_encoder(layout, _value_bins(max_abs))
    try:
        res = enc.encode(flat.ptr)
    finally:
        flat.free()
    return encode_streams_to_hic(res, g)


def _tables_to_arrays(table_payloads):
    from hiccup_b200 import codec
    return codec._tables_to_arrays(table_payloads)


def pyramid_of_file(hic):
    """The sub-band pyramid a wavelet HicImage's two shape payloads describe, read the way the reference reads them."""
    p = hic.payloads
    small, big = tuple(int(v) for v in p[12].numbers), tuple(int(v) for v in p[13].numbers)
    h, w = 2 * big[0], 2 * big[1]
    # codec.wavelet_decoded_subbands_shapes (codec.py:182-189): the level count is int(sqrt(big // small)) + 1 and
    # every level doubles exactly.  That formula is right for 2, 3 and 5 levels only; a 1- or 4-level file (or one
    # of inexact halvings) is mis-read by the reference itself, so it is refused here rather than mis-read too.
    if small[0] < 1 or small[1] < 1:
        raise ValueError("empty sub-band shape %r" % (small,))
    levels = int(np.sqrt(big[0] // small[0])) + 1
    if not 1 <= levels <= 5:
        raise ValueError("sub-band shapes %r .. %r imply %d levels" % (small, big, levels))
    g = _lib.wavelet_pyramid(h, w, levels)
    shapes = band_shapes(g)
    if shapes[0] != small or h % (1 << levels) or w % (1 << levels):
        raise ValueError("sub-band shapes %r .. %r are not a pyramid of exact halvings the reference's decoder reads "
                         "as it was written (codec.py:182-189)" % (small, big))
    return g


def decode_to_device_flat(hic, stream=None):
    """Entropy-decode a wavelet HicImage into the flat zigzag stream on the device."""
    assert hic.hic_type == model.Compression.HIC or getattr(hic.hic_type, "value", None) == "HIC"
    p = hic.payloads
    g = pyramid_of_file(hic)
    # stream order s = channel * 3 + kind; kind 0 (DC) is absent in flat mode
    empty = hicimage.PayloadStringP.from_rows([])
    tabs, bit_payloads = [], []
    for c in range(3):
        tabs += [empty, p[c], p[3 + c]]
        bit_payloads += [None, p[6 + c], p[9 + c]]
    rows, syms, lens, codes = _tables_to_arrays(tabs)
    offs, nbits, chunks, pos = [], [], [], 0
    for b in bit_payloads:
        if b is None:
            offs.append(0)
            nbits.append(0)
            continue
        framed = bytes(b.byte_stream)
        offs.append(pos)
        nbits.append(iohelper.payload_bit_count(framed))
        pad = (-len(framed)) % 4
        chunks.append(framed + b"\0" * pad)
        pos += len(framed) + pad
    data = np.frombuffer(b"".join(chunks) + b"\0" * 16, dtype=np.uint8)
    layout = _lib.layout_flat(1, int(g.len))
    flat = _lib.scratch(2 * _flat_elems(g) * 3)
    dec = entropy.cached_decoder(layout)
    try:
        from hiccup_b200 import codec
        codec._entropy_decode(dec, hic, rows, syms, lens, codes, data, offs, nbits, flat.ptr, stream)
    except Exception:
        flat.free()
        raise
    return flat, g


def wavelet_decode(hic: hicimage.HicImage) -> model.CompressedImage:
    settings.check_wavelet_supported()
    _lib.require_device()
    lib = _lib.load()
    flat, g = decode_to_device_flat(hic)
    d_bands = _lib.scratch(4 * int(g.len) * 3)
    _lib.check(lib.hic_wavelet_flat_to_bands_general(flat.ptr, 1, int(g.h), int(g.w), _levels_of(g), d_bands.ptr, None))
    arr = d_bands.download(np.int32, int(g.len) * 3).reshape(3, int(g.len))
    flat.free()
    d_bands.free()
    # the reference's decoded sub-bands are float64 (transform.izigzag builds them with np.zeros)
    return model.CompressedImage.from_dict(_split_bands(arr, g, np.float64))


def wavelet_decompression(channels: model.CompressedImage) -> np.ndarray:
    """Dequantise, inverse L-level db1, + 256, uint8 cast, YCrCb -> RGB.  The image is 2 ceil(h/2) x 2 ceil(w/2)
    as pywt.waverec2 returns it (compression.py:88-100); L comes from the number of sub-bands."""
    settings.check_wavelet_supported()
    _lib.require_device()
    lib = _lib.load()
    flat, g, _ = _bands_to_device_flat(channels)
    h, w, levels = int(g.h), int(g.w), _levels_of(g)
    rgb = _lib.scratch(h * w * 3)
    try:
        if levels == 3 and settings.WAVELET_SUBBAND_QUANTIZATION_MULTIPLIER == 1 and h % 8 == 0 and w % 8 == 0:
            _lib.check(lib.hic_wavelet_inverse(flat.ptr, 1, h, w, rgb.ptr, None))
        else:
            _run_general(levels, _lib.wavelet_work_bytes(1, h, w),
                         lambda params, work: lib.hic_wavelet_inverse_general(flat.ptr, 1, h, w, params, work, rgb.ptr, None))
        out = rgb.download(np.uint8, h * w * 3).reshape(h, w, 3)
    finally:
        flat.free()
        rgb.free()
    return out


def _run_general(levels, work_bytes, launch):
    """launch(params, work) -- a general entry on one image -- with a work area of work_bytes of its own, at `levels`
    and the multiplier of the settings now."""
    params = _lib.WaveletParams()
    params.levels, params.multiplier = levels, float(settings.WAVELET_SUBBAND_QUANTIZATION_MULTIPLIER)
    params.threshold, params.threshold_index = 0.0, -1
    work = _lib.scratch(work_bytes)
    try:
        _lib.check(launch(ctypes.byref(params), work.ptr))
        _lib.sync()
    finally:
        work.free()


def wavelet_scaled(hic: hicimage.HicImage, scale: int) -> np.ndarray:
    """The 1/scale image of a wavelet-mode file of L levels: (h / scale, w / scale, 3) uint8, scale = 2^k with
    1 <= k <= L.  Each sample is astype(uint8)(A_k * 2^-k + 256) of the running approximation A_k the full inverse holds
    after its first L - k levels -- the mean of each scale x scale tile of the unrounded full reconstruction -- and the
    three planes are converted to RGB as wavelet_decompression does (include/hiccup_b200.h, hic_wavelet_scaled_general,
    at the file's levels and the multiplier of the settings now).  The entropy decode is wavelet_decode's (restart
    records used when the file has them); the inverse transform stops k levels early and reads only the coarse
    sub-bands.  NotImplementedError for a DCT-mode file, ValueError for a bad scale or a pyramid pyramid_of_file
    refuses, all before any device work."""
    from hiccup_b200 import codec
    if codec._is_dct(hic):
        raise NotImplementedError("wavelet scaled decode works on wavelet-mode (HIC) files; this is a DCT-mode (JPEG) file")
    settings.check_wavelet_supported()
    g = pyramid_of_file(hic)
    h, w, levels = int(g.h), int(g.w), _levels_of(g)
    _lib.wavelet_scale_arg(scale, levels)
    scale = int(scale)
    lib = _lib.load()
    return _reduced_decode(hic, levels, (h // scale, w // scale, 3), _lib.wavelet_work_bytes(1, h, w),
                           lambda flat, params, work, rgb: lib.hic_wavelet_scaled_general(flat, 1, h, w, params, scale, work, rgb, None))


def wavelet_region(hic: hicimage.HicImage, top: int, left: int, height: int, width: int, scale: int = 1) -> np.ndarray:
    """One window of a wavelet-mode file of L levels: (height, width, 3) uint8.  At scale 1 it equals
    wavelet_decompression(wavelet_decode(hic))[top:top+height, left:left+width] bit for bit; at scale = 2^k,
    1 <= k <= L, the same window of wavelet_scaled(hic, scale), (top, left) in the coordinates of that image.  The
    entropy decode is wavelet_decode's (restart records used when the file has them); then only the window's dyadic
    parent rectangles of the sub-bands are read and inverse-transformed, with the full inverse's operations, straight
    into the window's pixels (include/hiccup_b200.h, hic_wavelet_region, at the file's levels and the multiplier of the
    settings now).  NotImplementedError for a DCT-mode file, ValueError for a bad scale, a window outside the 1/scale
    image or a pyramid pyramid_of_file refuses, all before any device work."""
    from hiccup_b200 import codec
    if codec._is_dct(hic):
        raise NotImplementedError("wavelet region decode works on wavelet-mode (HIC) files; this is a DCT-mode (JPEG) file")
    settings.check_wavelet_supported()
    g = pyramid_of_file(hic)
    h, w, levels = int(g.h), int(g.w), _levels_of(g)
    origin = _lib.wavelet_region_origins(h, w, levels, [(top, left)], (height, width), scale)
    scale, height, width = int(scale), int(height), int(width)
    lib = _lib.load()
    return _reduced_decode(hic, levels, (height, width, 3), origin.nbytes,
                           lambda flat, params, work, rgb: lib.hic_wavelet_region(flat, 1, h, w, params, scale, origin.ctypes.data,
                                                                                  height, width, work, origin.nbytes, rgb, None))


def _reduced_decode(hic, levels, shape, work_bytes, launch):
    """wavelet_decode's entropy stage into the flat stream on the device, then launch(flat, params, work, out) of a
    general entry into a uint8 image of `shape`, which is returned."""
    _lib.require_device()
    size = int(np.prod(shape))
    flat, _ = decode_to_device_flat(hic)
    rgb = _lib.scratch(size)
    try:
        _run_general(levels, work_bytes, lambda params, work: launch(flat.ptr, params, work, rgb.ptr))
        return rgb.download(np.uint8, size).reshape(shape)
    finally:
        flat.free()
        rgb.free()
