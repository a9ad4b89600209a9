"""Entropy-stage entry points, drop-in for reference hiccup/codec.py.

    jpeg_encode(compressed)     codec.py:275-334     jpeg_decode(hic)     codec.py:337-426
    wavelet_encode(compressed)  codec.py:116-163     wavelet_decode(hic)  codec.py:199-239

Same argument meaning and return types (`HicImage` with the reference's payload order).  DC
differencing, run-length coding, histogramming, bit packing and their inverses run in the CUDA
kernels behind include/hiccup_b200.h; the Huffman trees are built on the host by an exact replay of
the reference's heapq construction (csrc/hic_huffman.cuh).
"""
import numpy as np

from hiccup_b200 import _lib, compression, entropy, hicimage, iohelper, model, settings

CHANNELS = ("lum", "cr", "cb")


def _pick_value_bins(max_abs):
    """Smallest power-of-two bin count whose half covers DC differences (up to 2 * max_abs)."""
    need = 2 * int(max_abs) + 2
    bins = entropy.DEFAULT_VALUE_BINS
    while bins // 2 < need:
        bins *= 2
    if bins > 65536:
        raise ValueError("coefficients up to %d do not fit the int16 symbol path" % max_abs)
    return bins


def _integral_planes(planes):
    out = []
    for a in planes:
        a = np.asarray(a)
        if a.dtype.kind == "f":
            r = np.rint(a)
            if not np.array_equal(r, a):
                raise NotImplementedError("non-integral coefficients are not on the CUDA entropy path")
            a = r
        out.append(a)
    return out


def _symbol_types(dtype):
    """Python types the reference's symbols have in the pickled tables (SURVEY hard part 3): DC
    symbols keep the plane's numpy scalar type (codec.py:47-52 on ndarray elements); run-length
    values pass through ndarray.tolist() (transform.py:264) -> Python int/float; zero counts are
    Python ints."""
    dc_type = np.dtype(dtype).type
    ac_type = float if np.dtype(dtype).kind == "f" else int
    return dc_type, ac_type


def jpeg_encode(compressed: model.CompressedImage, restarts: bool = False) -> hicimage.HicImage:
    """restarts=True appends the restart records of the nine bit strings as an extension entry (hicimage.RestartP):
    the reference's reader ignores it, this package's decoder then skips the synchronisation passes."""
    hic = _jpeg_encode(compressed)
    return add_restart_records(hic) if restarts else hic


def _jpeg_encode(compressed: model.CompressedImage) -> hicimage.HicImage:
    settings.check_supported()
    _lib.require_device()
    d = compressed.as_dict if hasattr(compressed, "as_dict") else model.CompressedImage.as_dict.fget(compressed)
    src_dtype = np.asarray(d["lum"]).dtype
    planes = _integral_planes([d[c] for c in CHANNELS])
    max_abs = max(int(np.abs(p).max()) if p.size else 0 for p in planes)
    bins = _pick_value_bins(max_abs)
    comp = model.CompressedImage(*planes)
    coef, g = compression.planes_to_device_blocks(comp)
    layout = _lib.layout_dct(1, g.h, g.w)
    enc = entropy.cached_encoder(layout, bins)
    try:
        res = enc.encode(coef.ptr)
    finally:
        coef.free()
    dc_type, ac_type = _symbol_types(src_dtype)
    tables, bits = [], []
    for kind in (entropy.KIND_DC, entropy.KIND_VALUE, entropy.KIND_LENGTH):
        for c in range(3):
            s = c * 3 + kind
            conv = dc_type if kind == entropy.KIND_DC else (ac_type if kind == entropy.KIND_VALUE else int)
            if conv is int or conv is np.int32:       # the usual case: the table stays three arrays (hicimage.from_arrays)
                sym, lens, codes = res.stream_rows(s)
                tables.append(hicimage.PayloadStringP.from_arrays(sym, lens, codes, conv is np.int32))
            else:
                tables.append(hicimage.PayloadStringP.from_rows([(conv(sym), code) for sym, code in res.table(s)]))
            bits.append(hicimage.BitStringP.from_framed(res.framed(s)))
    lum_shape = tuple(int(v) for v in planes[0].shape)
    cr_shape = tuple(int(v) for v in planes[1].shape)
    payloads = tables + bits + [hicimage.TupP(*lum_shape), hicimage.TupP(*cr_shape)]
    return hicimage.HicImage.jpeg_image(payloads)


def _tables_to_arrays(table_payloads):
    rows, syms, lens, codes = [], [], [], []
    for t in table_payloads:
        arrays = t.arrays() if hasattr(t, "arrays") else None
        if arrays is not None:
            rows.append(int(arrays[0].size))
            syms.append(arrays[0])
            lens.append(arrays[1])
            codes.append(arrays[2])
            continue
        r = t.rows if hasattr(t, "rows") else [p.numbers for p in t.payloads]
        rows.append(len(r))
        syms.append(np.array([int(sym) for sym, _ in r], np.int32))
        lens.append(np.array([len(code) for _, code in r], np.uint8))
        codes.append(np.array([int(code, 2) for _, code in r], np.uint64))
    cat = lambda xs, dt: np.concatenate(xs).astype(dt, copy=False) if xs else np.zeros(0, dt)
    return rows, cat(syms, np.int32), cat(lens, np.uint8), cat(codes, np.uint64)


def _gather_payload_bytes(bit_payloads):
    """Lay the framed payloads out 4-byte aligned in one host array."""
    offs, nbits, chunks, pos = [], [], [], 0
    for b in bit_payloads:
        framed = bytes(b.byte_stream)
        offs.append(pos)
        nbits.append(iohelper.payload_bit_count(framed))
        pad = (-len(framed)) % 4
        chunks.append(framed + b"\0" * pad)
        pos += len(framed) + pad
    data = np.frombuffer(b"".join(chunks) + b"\0" * 16, dtype=np.uint8)
    return data, offs, nbits


def _stream_order(hic):
    """File payload index of the table / bit string of every stream s of the entropy stage, (tables, bits);
    None where the stream does not exist (the DC streams of a wavelet file)."""
    if _is_dct(hic):       # reference order is (kind, channel); stream order is s = channel * 3 + kind
        order = [kind * 3 + c for c in range(3) for kind in range(3)]
        return order, [9 + i for i in order], 9
    tabs, bits = [], []
    for c in range(3):     # kind 0 (DC) is absent in flat mode
        tabs += [None, c, 3 + c]
        bits += [None, 6 + c, 9 + c]
    return tabs, bits, 6


def _records_in_stream_order(hic, nbits, kinds=(0, 1, 2)):
    """The file's restart records re-ordered to stream order and concatenated, or None when the file has none
    (or they do not fit its bit strings: the extension is advisory, the decoder then synchronises by itself).
    kinds: the symbol kinds whose records are wanted (the DC-only decode takes kind 0 alone)."""
    ext = getattr(hic, "restarts", None)
    if ext is None:
        return None
    _, bits, first = _stream_order(hic)
    n_bits = len(bits) - bits.count(None)
    if len(ext.records) != n_bits:
        return None
    want = entropy.EntropyDecoder.subsequences(nbits)
    offs, cnts = [], []
    for s, i in enumerate(bits):
        if i is None or s % 3 not in kinds:
            continue
        off, cnt = ext.records[i - first]
        if off.size != want[s] or cnt.size != want[s]:
            return None
        offs.append(off)
        cnts.append(cnt)
    return np.concatenate(offs) if offs else np.zeros(0, np.uint8), np.concatenate(cnts) if cnts else np.zeros(0, np.uint8)


def _entropy_decode(dec, hic, rows, syms, lens, codes, data, offs, nbits, d_coef, stream=None):
    records = _records_in_stream_order(hic, nbits)
    if records is not None:
        try:
            dec.decode(rows, syms, lens, codes, data, offs, nbits, d_coef, stream, restarts=records)
            return True
        except _lib.HicError:
            pass           # records that do not belong to the streams: decode the long way (and fail there if the streams are bad)
    dec.decode(rows, syms, lens, codes, data, offs, nbits, d_coef, stream)
    return False


def add_restart_records(hic: hicimage.HicImage) -> hicimage.HicImage:
    """A copy of `hic` carrying the restart records of its bit strings (an extension entry the reference's reader
    never reads): D1's synchronisation passes run once, here, instead of at every decode."""
    _lib.require_device()
    p = hic.payloads
    tabs, bits, first = _stream_order(hic)
    empty = hicimage.PayloadStringP.from_rows([])
    rows, syms, lens, codes = _tables_to_arrays([empty if i is None else p[i] for i in tabs])
    jpeg = first == 9
    offs, nbits, chunks, pos = [], [], [], 0
    for i in bits:
        if i is None:
            offs.append(0)
            nbits.append(0)
            continue
        framed = bytes(p[i].byte_stream)
        offs.append(pos)
        nbits.append(iohelper.payload_bit_count(framed))
        pad = (-len(framed)) % 4
        chunks.append(framed + b"\0" * pad)
        pos += len(framed) + pad
    data = np.frombuffer(b"".join(chunks) + b"\0" * 16, dtype=np.uint8)
    if jpeg:
        h, w = (int(v) for v in p[18].numbers)
        layout = _lib.layout_dct(1, h, w)
    else:
        from hiccup_b200 import wavelet
        layout = _lib.layout_flat(1, int(wavelet.pyramid_of_file(hic).len))
    dec = entropy.cached_decoder(layout)
    off, cnt = dec.decode(rows, syms, lens, codes, data, offs, nbits, None, sync_only=True)
    n_sub = entropy.EntropyDecoder.subsequences(nbits)
    records, at = {}, 0
    for s, i in enumerate(bits):
        if i is None:
            continue
        records[i - first] = (off[at:at + n_sub[s]], cnt[at:at + n_sub[s]])
        at += n_sub[s]
    ext = hicimage.RestartP([records[k] for k in sorted(records)])
    others = [e for e in hic.extensions if not isinstance(e, hicimage.RestartP)]
    return hicimage.HicImage(hic.hic_type, hic.settings, list(p), others + [ext])


def _is_dct(hic):
    return hic.hic_type == model.Compression.JPEG or getattr(hic.hic_type, "value", None) == "JPEG"


def _require_dct(hic, what):
    if not _is_dct(hic):
        raise NotImplementedError("%s works on DCT-mode (JPEG) files; this is a wavelet (HIC) file" % what)


def _dct_header(hic):
    """(payloads, h, w, geometry) of a DCT-mode file; ValueError when its chroma shape does not belong to its luminance
    shape."""
    p = hic.payloads
    lum_shape, cr_shape = tuple(p[18].numbers), tuple(p[19].numbers)
    h, w = int(lum_shape[0]), int(lum_shape[1])
    g = _lib.geometry(h, w)
    if (g.hc, g.wc) != (int(cr_shape[0]), int(cr_shape[1])):
        raise ValueError("chroma shape %r does not belong to luminance shape %r" % (cr_shape, lum_shape))
    return p, h, w, g


def _decode_coefficients(hic, h, w, d_coef):
    """D1-D3 of all nine streams of a DCT-mode file into d_coef ([blocks][64] int16), with the file's restart records
    when they fit."""
    p = hic.payloads
    tabs, bits, _ = _stream_order(hic)
    rows, syms, lens, codes = _tables_to_arrays([p[i] for i in tabs])
    data, offs, nbits = _gather_payload_bytes([p[i] for i in bits])
    _entropy_decode(entropy.cached_decoder(_lib.layout_dct(1, h, w)), hic, rows, syms, lens, codes, data, offs, nbits, d_coef)


def jpeg_decode(hic: hicimage.HicImage) -> model.CompressedImage:
    settings.check_supported()
    _lib.require_device()
    assert _is_dct(hic)
    _, h, w, g = _dct_header(hic)
    coef = _lib.scratch(g.blocks_per_image * 128)
    lib = _lib.load()
    try:
        _decode_coefficients(hic, h, w, coef.ptr)
        lum = _lib.scratch(4 * h * w)
        cr = _lib.scratch(4 * g.hc * g.wc)
        cb = _lib.scratch(4 * g.hc * g.wc)
        _lib.check(lib.hic_blocks_to_planes(coef.ptr, 1, h, w, lum.ptr, cr.ptr, cb.ptr, None))
        # the reference's decoded planes are float64 (transform.izigzag builds them with np.zeros)
        out = model.CompressedImage(lum.download(np.int32, h * w).reshape(h, w).astype(np.float64),
                                    cr.download(np.int32, g.hc * g.wc).reshape(g.hc, g.wc).astype(np.float64),
                                    cb.download(np.int32, g.hc * g.wc).reshape(g.hc, g.wc).astype(np.float64))
        for b in (lum, cr, cb):
            b.free()
    finally:
        coef.free()
    return out


def jpeg_thumbnail(hic: hicimage.HicImage) -> np.ndarray:
    """The 1/8-scale preview of a DCT-mode file: (th, tw, 3) uint8, one pixel per 8x8 tile of what jpeg_decode +
    compression.jpeg_decompression return (th = ceil(out_h / 8)), from the three DC streams alone (hic_dct_thumbnail).
    Only the DC tables and DC bit strings go to the device; the file's restart records of the DC streams are used
    when it has them."""
    # a wavelet file has no DC streams: its coarse band would need a prefix decode of the value and length streams
    _require_dct(hic, "thumbnail decode")
    settings.check_supported()
    _lib.require_device()
    _, h, w, g = _dct_header(hic)
    lib = _lib.load()
    return _reduced_decode(hic, h, w, g, _lib.thumbnail_shape(h, w) + (3,),
                           lambda dc, out: lib.hic_dct_thumbnail(dc, 1, h, w, out, None), dc_only=True)


def _decode_dc(hic, h, w, d_dc):
    """The DC-only entropy decode of a DCT-mode file into d_dc, one int16 per block: only the DC tables and DC bit
    strings go to the device, with the file's restart records of the DC streams when it has them."""
    p = hic.payloads
    # stream order s = channel * 3 + kind; the DC table / bit string of channel c is payload c / 9 + c
    rows, syms, lens, codes = _tables_to_arrays([p[c] for c in range(3)])
    index = np.zeros((9, 2), np.uint32)
    index[0::3, 1] = rows
    index[0::3, 0] = np.concatenate(([0], np.cumsum(rows)[:-1]))
    packed = (lens.astype(np.uint64) << np.uint64(58)) | (codes & entropy.CODE_MASK)
    data, offs3, nbits3 = _gather_payload_bytes([p[9 + c] for c in range(3)])
    offs, nbits = np.zeros(9, np.uint64), np.zeros(9, np.uint64)
    offs[0::3], nbits[0::3] = offs3, nbits3
    records = _records_in_stream_order(hic, nbits, kinds=(entropy.KIND_DC,))
    dec = entropy.cached_decoder(_lib.layout_dct(1, h, w))
    dec.decode_dc(index, syms, packed, data, offs, nbits, d_dc, restarts=records)


def _reduced_decode(hic, h, w, g, shape, launch, scratch=(), dc_only=False):
    """jpeg_decode's entropy stage into a device buffer -- all nine streams into coefficient blocks, or (dc_only) the DC
    streams alone into one int16 per block (_decode_dc) -- then launch(src, out, *scratch pointers) with that buffer, a
    uint8 image of `shape` and one scratch buffer per byte count in `scratch`.  The image is returned."""
    size = int(np.prod(shape))
    bufs = [_lib.scratch(g.blocks_per_image * (2 if dc_only else 128)), _lib.scratch(size)]
    bufs += [_lib.scratch(b) for b in scratch]
    try:
        (_decode_dc if dc_only else _decode_coefficients)(hic, h, w, bufs[0].ptr)
        _lib.check(launch(*(b.ptr for b in bufs)))
        return bufs[1].download(np.uint8, size).reshape(shape)
    finally:
        for b in bufs:
            b.free()


def _tie_stage(entry, h, w, params, sizes):
    """(launch, scratch) of _reduced_decode for hic_dct_region, hic_dct_scaled or hic_dct_scaled_region, called as
    (coef, 1, h, w, *params, work, work bytes, ties, tie capacity, stats, out, stream) with the (work bytes, tie
    capacity) of `sizes`."""
    work_bytes, tie_cap = sizes

    def launch(coef, out, work, ties, stats):
        return entry(coef, 1, h, w, *params, work, work_bytes, ties, tie_cap, stats, out, None)
    return launch, (work_bytes, tie_cap * _lib.TIE_RECORD_BYTES, 4 * _lib.TIE_STATS)


def jpeg_region(hic: hicimage.HicImage, top: int, left: int, height: int, width: int, scale: int = 1) -> np.ndarray:
    """One window of a DCT-mode file: (height, width, 3) uint8.  At scale 1 it is the window of the full-resolution
    image, equal to compression.jpeg_decompression(jpeg_decode(hic))[top:top+height, left:left+width] bit for bit: the
    entropy decode is jpeg_decode's (restart records used when the file has them); then only the blocks the window
    reads are inverse-transformed and only its pixels upsampled and converted (hic_dct_region).  At scale 2 or 4 the
    window is one of jpeg_scaled(hic, scale), equal to its crop, with only the window's blocks reduced-transformed
    (hic_dct_scaled_region); at scale 8 one of jpeg_thumbnail(hic), from the DC streams alone
    (hic_dct_thumbnail_region).  (top, left) is in the coordinates of the 1/scale image.  ValueError for a scale other
    than 1, 2, 4 or 8 or a window outside the 1/scale image, NotImplementedError for a wavelet file, all before any
    device work."""
    _require_dct(hic, "region decode")
    scale = _lib.region_scale_arg(scale)
    _, h, w, g = _dct_header(hic)
    origin = _lib.region_origins(h, w, [(top, left)], (height, width), scale)
    settings.check_supported()
    _lib.require_device()
    height, width = int(height), int(width)
    lib, o = _lib.load(), origin.ctypes.data
    if scale == 1:
        launch, scratch = _tie_stage(lib.hic_dct_region, h, w, (o, height, width), _lib.region_sizes(1, h, w, height, width))
    elif scale != 8:
        launch, scratch = _tie_stage(lib.hic_dct_scaled_region, h, w, (scale, o, height, width),
                                     _lib.scaled_region_sizes(1, h, w, scale, height, width))
    else:
        work_bytes = _lib.scaled_region_sizes(1, h, w, 8, height, width)[0]
        scratch = (work_bytes,)

        def launch(dc, out, work):
            return lib.hic_dct_thumbnail_region(dc, 1, h, w, o, height, width, work, work_bytes, out, None)
    return _reduced_decode(hic, h, w, g, (height, width, 3), launch, scratch, dc_only=scale == 8)


def jpeg_scaled(hic: hicimage.HicImage, scale: int) -> np.ndarray:
    """The 1/2- or 1/4-scale image of a DCT-mode file: (ceil(out_h / scale), ceil(out_w / scale), 3) uint8.  Each
    8x8 block gives an m x m tile (m = 8 / scale) by a reduced inverse transform of its low-frequency m x m
    coefficients, the mean of each scale x scale tile of its IDCT, with the exact float64 definition of
    hic_dct_scaled; the chroma planes are upsampled and converted with the full decode's integer rules.  The
    entropy decode is jpeg_decode's (restart records used when the file has them).  ValueError for a scale other
    than 2 or 4 (1/8 is jpeg_thumbnail), NotImplementedError for a wavelet file, both before any device work."""
    _require_dct(hic, "scaled decode")
    scale = _lib.scale_arg(scale)
    _, h, w, g = _dct_header(hic)
    settings.check_supported()
    _lib.require_device()
    return _reduced_decode(hic, h, w, g, _lib.scaled_shape(h, w, scale) + (3,),
                           *_tie_stage(_lib.load().hic_dct_scaled, h, w, (scale,), _lib.scaled_sizes(1, h, w, scale)))


def wavelet_encode(compressed: model.CompressedImage, restarts: bool = False) -> hicimage.HicImage:
    from hiccup_b200 import wavelet
    hic = wavelet.wavelet_encode(compressed)
    return add_restart_records(hic) if restarts else hic


def wavelet_decode(hic: hicimage.HicImage) -> model.CompressedImage:
    from hiccup_b200 import wavelet
    return wavelet.wavelet_decode(hic)


def wavelet_scaled(hic: hicimage.HicImage, scale: int) -> np.ndarray:
    from hiccup_b200 import wavelet
    return wavelet.wavelet_scaled(hic, scale)


def wavelet_region(hic: hicimage.HicImage, top: int, left: int, height: int, width: int, scale: int = 1) -> np.ndarray:
    from hiccup_b200 import wavelet
    return wavelet.wavelet_region(hic, top, left, height, width, scale)
