"""Thumbnail decode on the GPU: the DC-only entropy decode (hic_decode_run_dc) and the thumbnail kernel
(hic_dct_thumbnail) give, bit for bit, the oracle thumbnail of tests/thumbnail_oracle.py -- from the reference's own
`.hic` bytes, from codec-encoded odd sizes, from DC values that wrap, with and without restart records, for whole
batches and through the file driver -- and never read the AC streams."""
import os
import pickle

import numpy as np
import pytest

from oracle import hiccup_oracle as orc
from tests import thumbnail_oracle as tho
from tests.conftest import load_golden
from tests.reduced_helpers import DCT_GOLDENS, kernels_of, planes

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", DCT_GOLDENS)
def test_reference_files(name):
    from hiccup_b200 import codec, hicimage
    g = load_golden(name)
    hi = hicimage.HicImage.from_bytes(pickle.loads(g["hic"].tobytes()))
    got, kernels = kernels_of(lambda: codec.jpeg_thumbnail(hi))
    want = tho.jpeg_thumbnail({ch: g["coef_" + ch] for ch in orc.CHANNELS})
    assert got.shape == want.shape and np.array_equal(got, want)
    assert "thumbnail_kernel" in kernels and "validate_dc_kernel" in kernels
    assert not kernels & {"expand_scatter_kernel", "inverse_kernel", "upsample_colour_kernel", "validate_kernel"}


@pytest.mark.parametrize("shape", [(40, 41), (41, 40), (33, 47), (26, 40), (40, 40), (41, 41), (9, 17), (2, 2)])
def test_odd_sizes(shape):
    from hiccup_b200 import codec, compression
    rgb = orc.synthetic_image(shape[0], shape[1], 300 + shape[0] * 7 + shape[1])
    comp = compression.jpeg_compression(rgb)
    got = codec.jpeg_thumbnail(codec.jpeg_encode(comp))
    assert np.array_equal(got, tho.jpeg_thumbnail(planes(comp)))


def test_dc_values_that_wrap():
    """DC terms whose DC-only block leaves 0..255 (truncation toward zero, then the uint8 wrap), in all three planes."""
    from hiccup_b200 import codec, model
    rng = np.random.default_rng(17)
    h, w = 83, 122
    planes = {}
    for ch, shape in (("lum", (h, w)), ("cr", (h // 2, w // 2)), ("cb", (h // 2, w // 2))):
        p = rng.integers(-3, 4, shape).astype(np.int32) * (rng.random(shape) < 0.2)
        p[::8, ::8] = rng.integers(-6000, 6000, p[::8, ::8].shape)
        p[0, 0], p[0, 8] = 2041, -2049                                  # just past each end on luminance
        planes[ch] = p.astype(np.int32)
    for ch in orc.CHANNELS:                                              # q T00 / 256 + 128 leaves 0..255 on both sides
        q = tho.dc_terms(planes[ch])
        assert (q < -2048).any() and (q > 2040).any()
    hi = codec.jpeg_encode(model.CompressedImage(planes["lum"], planes["cr"], planes["cb"]))
    assert np.array_equal(codec.jpeg_thumbnail(hi), tho.jpeg_thumbnail(planes))


def test_restart_records():
    from hiccup_b200 import codec, compression, hicimage
    rgb = orc.synthetic_image(426, 640, 2000)
    comp = compression.jpeg_compression(rgb)
    want = tho.jpeg_thumbnail(planes(comp))
    plain = codec.jpeg_encode(comp)
    ext = hicimage.HicImage.from_bytes(codec.jpeg_encode(comp, restarts=True).byte_stream())
    got, k_plain = kernels_of(lambda: codec.jpeg_thumbnail(plain))
    assert np.array_equal(got, want) and "huffman_sync_kernel" in k_plain
    got, k_ext = kernels_of(lambda: codec.jpeg_thumbnail(ext))
    assert np.array_equal(got, want)
    assert "restart_load_kernel" in k_ext and "huffman_sync_kernel" not in k_ext
    # records that do not belong: the write pass finds out and the decode synchronises by itself
    bad = [(np.zeros_like(o), np.ones_like(c)) for o, c in ext.restarts.records]
    hx = hicimage.HicImage(ext.hic_type, ext.settings, ext.payloads, [hicimage.RestartP(bad)])
    got, kernels = kernels_of(lambda: codec.jpeg_thumbnail(hx))
    assert np.array_equal(got, want) and "huffman_sync_kernel" in kernels
    # records of the wrong size are not even tried
    short = [(o[:-1], c[:-1]) for o, c in ext.restarts.records]
    hy = hicimage.HicImage(ext.hic_type, ext.settings, ext.payloads, [hicimage.RestartP(short)])
    got, kernels = kernels_of(lambda: codec.jpeg_thumbnail(hy))
    assert np.array_equal(got, want) and "restart_load_kernel" not in kernels


def _dc_decode_thumbnail(h, w, index, symbols, packed, data, byte_off, nbits, data_bytes):
    from hiccup_b200 import _lib, entropy
    lib = _lib.load()
    dec = entropy.EntropyDecoder(_lib.layout_dct(1, h, w))
    g = _lib.geometry(h, w)
    th, tw = _lib.thumbnail_shape(h, w)
    d_data = _lib.DeviceBuffer(data.nbytes + 16)
    d_dc = _lib.DeviceBuffer(2 * g.blocks_per_image)
    out = _lib.DeviceBuffer(3 * th * tw)
    try:
        d_data.upload(data)
        _lib.check(lib.hic_decode_set_tables_packed(dec.plan, np.ascontiguousarray(index, np.uint32).ctypes.data,
                                                    symbols.ctypes.data, packed.ctypes.data, int(symbols.size), None))
        _lib.check(lib.hic_decode_set_data_bytes(dec.plan, int(data_bytes)))
        dec.run_dc(d_data.ptr, byte_off, nbits, d_dc.ptr)
        _lib.check(lib.hic_dct_thumbnail(d_dc.ptr, 1, h, w, out.ptr, None))
        return out.download(np.uint8, 3 * th * tw).reshape(th, tw, 3)
    finally:
        for b in (d_data, d_dc, out):
            b.free()
        dec.close()


def test_ac_streams_are_never_read():
    """All nine tables installed, the AC streams' bytes overwritten with random data and their offsets past the
    data-bytes bound, which covers the DC streams alone: the thumbnail does not change."""
    from hiccup_b200 import codec, compression, entropy, iohelper
    rgb = orc.synthetic_image(96, 136, 44)
    comp = compression.jpeg_compression(rgb)
    hi = codec.jpeg_encode(comp)
    want = tho.jpeg_thumbnail(planes(comp))
    p = hi.payloads
    order = [kind * 3 + c for c in range(3) for kind in range(3)]          # stream s = channel * 3 + kind
    rows, syms, lens, codes = codec._tables_to_arrays([p[i] for i in order])
    index = np.stack([np.concatenate(([0], np.cumsum(rows)[:-1])), rows], 1).astype(np.uint32)
    packed = (lens.astype(np.uint64) << np.uint64(58)) | (codes & entropy.CODE_MASK)
    framed = [bytes(p[9 + i].byte_stream) for i in order]
    byte_off, nbits, pos = np.zeros(9, np.uint64), np.zeros(9, np.uint64), 0
    dc_part = b""
    for s in range(0, 9, 3):
        byte_off[s], nbits[s] = pos, iohelper.payload_bit_count(framed[s])
        chunk = framed[s] + b"\0" * ((-len(framed[s])) % 4)
        dc_part += chunk
        pos += len(chunk)
    rng = np.random.default_rng(3)
    ac_part = rng.integers(0, 256, sum(len(f) + 8 for f in framed), dtype=np.uint8).tobytes()
    for s in range(9):
        if s % 3:
            byte_off[s] = pos + 4 * s                                        # inside the random bytes, past the bound
            nbits[s] = 8 * (len(framed[s]) - 1)
    data = np.frombuffer(dc_part + ac_part + b"\0" * 16, np.uint8)
    got = _dc_decode_thumbnail(96, 136, index, syms, packed, data, byte_off, nbits, data_bytes=len(dc_part))
    assert np.array_equal(got, want)
    # the same streams with the AC tables gone (zero rows): the DC-only decode needs nothing else
    index_dc = index.copy()
    index_dc[[s for s in range(9) if s % 3], 1] = 0
    got = _dc_decode_thumbnail(96, 136, index_dc, syms, packed, data, byte_off, nbits, data_bytes=len(dc_part))
    assert np.array_equal(got, want)


def test_short_dc_stream_is_corrupt():
    """A DC bit string that holds one symbol fewer than the channel has blocks is HIC_ERR_CORRUPT, not a picture."""
    from hiccup_b200 import _lib, codec, compression, hicimage
    rgb = orc.synthetic_image(64, 96, 45)
    comp = compression.jpeg_compression(rgb)
    hi = codec.jpeg_encode(comp)
    streams = orc.jpeg_streams(planes(comp))
    for c, ch in enumerate(orc.CHANNELS):
        table = [(int(sym), code) for sym, code in hi.payloads[c].rows]
        bits = orc.huffman_encode_bits(streams["dc"][ch][:-1], table)
        payloads = list(hi.payloads)
        payloads[9 + c] = hicimage.BitStringP.from_framed(orc.padded_bits_to_bytes(bits))
        cut = hicimage.HicImage(hi.hic_type, hi.settings, payloads, [])
        with pytest.raises(_lib.HicError, match="error -4"):
            codec.jpeg_thumbnail(cut)
    assert np.array_equal(codec.jpeg_thumbnail(hi), tho.jpeg_thumbnail(planes(comp)))


@pytest.mark.parametrize("n,h,w", [(5, 40, 41), (3, 33, 47), (4, 64, 96)])
def test_batch(n, h, w):
    from hiccup_b200 import codec
    from hiccup_b200.batch import DctBatchCodec
    rgb = np.stack([orc.synthetic_image(h, w, 500 + i) for i in range(n)])
    bc = DctBatchCodec(n, h, w)
    try:
        enc = bc.encode(rgb)
        want = np.stack([codec.jpeg_thumbnail(hi) for hi in bc.hic_images(enc)])
        assert bc.thumbnail_shape == want.shape
        assert np.array_equal(bc.thumbnails(enc), want)
        out = np.zeros(bc.thumbnail_shape, np.uint8)
        assert bc.thumbnails(enc, out=out) is not None and np.array_equal(out, want)
        bc.thumbnails_device()
        assert np.array_equal(bc.fetch_thumbnails(), want)
        assert np.array_equal(bc.thumbnails(bc.streams_from_files(bc.hic_files(enc))), want)
        for i in range(n):
            assert np.array_equal(want[i], tho.jpeg_thumbnail(orc.jpeg_compression(rgb[i])))
    finally:
        bc.close()


def test_c2_batch(tmp_path):
    """1024 x 640x426 (the benchmark's C2 batch): thumbnails from the encoder's device output, from the host streams
    and from the written `.hic` files agree; eight seeded images equal codec.jpeg_thumbnail and the oracle."""
    from hiccup_b200 import codec
    from hiccup_b200.batch import DctBatchCodec
    n, h, w = 1024, 426, 640
    base = np.stack([orc.synthetic_image(h, w, 2000 + i) for i in range(16)])
    rgb = np.ascontiguousarray(base[np.arange(n) % 16])
    rgb[:, 0, :, 0] = (np.arange(n) // 16).astype(np.uint8)[:, None]        # 1024 distinct images
    bc = DctBatchCodec(n, h, w)
    try:
        enc = bc.encode(rgb)
        got = bc.thumbnails(enc).copy()
        bc.thumbnails_device()
        assert np.array_equal(bc.fetch_thumbnails(), got)
        paths = [os.path.join(tmp_path, "%04d.hic" % i) for i in range(n)]
        bc.write_files(enc, paths)
        assert np.array_equal(bc.thumbnails(bc.read_files(paths)), got)
        pick = np.random.default_rng(2024).choice(n, 8, replace=False)
        his = bc.hic_images(enc, images=[int(i) for i in pick])
        for i, hi in zip(pick, his):
            assert np.array_equal(got[i], codec.jpeg_thumbnail(hi))
            assert np.array_equal(got[i], tho.jpeg_thumbnail(orc.jpeg_compression(rgb[i])))
    finally:
        bc.close()


def test_file_driver(tmp_path):
    import cv2
    from hiccup_b200 import model, run
    srcs = []
    for i, (h, w) in enumerate([(40, 41), (40, 41), (72, 96), (40, 41)]):
        p = os.path.join(tmp_path, "img%d.png" % i)
        cv2.imwrite(p, orc.synthetic_image(h, w, 70 + i))
        srcs.append(p)
    files = [run.compress(p, str(tmp_path), model.Compression.JPEG, restarts=(i == 1)) for i, p in enumerate(srcs)]
    out_dir = os.path.join(tmp_path, "thumbs")
    os.makedirs(out_dir)
    many = run.decompress_many(files, save_dir=out_dir, max_batch=2, thumbnail=True)
    for f, t in zip(files, many):
        one = run.decompress(f, thumbnail=True)
        assert np.array_equal(t, one)
        assert np.array_equal(cv2.imread(os.path.join(out_dir, os.path.basename(f) + ".thumb.png")), one)
    run.main(["-d", files[2], "-t", "-o", out_dir])
    assert os.path.exists(os.path.join(out_dir, os.path.basename(files[2]) + ".thumb.png"))
