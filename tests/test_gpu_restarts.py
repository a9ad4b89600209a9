"""Restart records (SURVEY section 8(f) rank 4): an extension entry appended to a `.hic` file that lets the decoder
skip D1's synchronisation passes.  The reference's 21 / 15 entries stay byte-identical, the decoded planes are the
same with and without the records, and records that do not belong to the streams never change the result."""
import numpy as np
import pytest

from oracle import hiccup_oracle as orc
from tests.reduced_helpers import kernels_of

pytestmark = pytest.mark.gpu


def _same_planes(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a.as_dict.values(), b.as_dict.values()))


@pytest.mark.parametrize("shape,seed", [((64, 96), 1), ((426, 640), 2), ((720, 1280), 3)])
def test_dct_file_with_restart_records(shape, seed):
    from hiccup_b200 import codec, compression, hicimage
    rgb = orc.synthetic_image(shape[0], shape[1], 50 + seed)
    comp = compression.jpeg_compression(rgb)
    plain = codec.jpeg_encode(comp)
    ext = codec.jpeg_encode(comp, restarts=True)
    assert ext.byte_stream()[:21] == plain.byte_stream() and len(ext.byte_stream()) == 22
    rec = ext.restarts
    assert rec is not None and len(rec.records) == 9
    for (off, cnt), p in zip(rec.records, ext.payloads[9:18]):
        n_sub = (8 + p.bit_count + 127) // 128
        assert off.size == cnt.size == n_sub
        assert int(cnt.astype(np.int64).sum()) > 0 and off.max(initial=0) < 58 and cnt.max(initial=0) <= 128
    back = hicimage.HicImage.from_bytes(ext.byte_stream())           # through the wire
    want, k_plain = kernels_of(lambda: codec.jpeg_decode(plain))
    got, k_ext = kernels_of(lambda: codec.jpeg_decode(back))
    assert _same_planes(got, want)
    assert "huffman_sync_kernel" in k_plain and "huffman_sync_kernel" not in k_ext and "huffman_resync_kernel" not in k_ext
    assert "restart_load_kernel" in k_ext
    # symbol counts of the records are the streams' symbol counts: DC streams hold one symbol per block
    g_blocks = [-(-shape[0] // 8) * -(-shape[1] // 8), -(-(shape[0] // 2) // 8) * -(-(shape[1] // 2) // 8)]
    assert int(rec.records[0][1].astype(np.int64).sum()) == g_blocks[0]
    assert int(rec.records[1][1].astype(np.int64).sum()) == g_blocks[1]


def test_records_that_do_not_fit_are_ignored():
    from hiccup_b200 import codec, compression, hicimage
    rgb = orc.synthetic_image(128, 192, 9)
    comp = compression.jpeg_compression(rgb)
    ext = codec.jpeg_encode(comp, restarts=True)
    want = codec.jpeg_decode(codec.jpeg_encode(comp))
    # (a) wrong contents: the write pass finds out, the decoder synchronises by itself
    bad = [(np.zeros_like(o), np.ones_like(c)) for o, c in ext.restarts.records]
    hx = hicimage.HicImage(ext.hic_type, ext.settings, ext.payloads, [hicimage.RestartP(bad)])
    got, kernels = kernels_of(lambda: codec.jpeg_decode(hx))
    assert _same_planes(got, want) and "huffman_sync_kernel" in kernels
    # (b) wrong sizes: not even tried
    short = [(o[:-1], c[:-1]) for o, c in ext.restarts.records]
    hy = hicimage.HicImage(ext.hic_type, ext.settings, ext.payloads, [hicimage.RestartP(short)])
    got, kernels = kernels_of(lambda: codec.jpeg_decode(hy))
    assert _same_planes(got, want) and "restart_load_kernel" not in kernels


def test_wavelet_file_with_restart_records():
    from hiccup_b200 import codec, compression, hicimage
    rgb = orc.synthetic_image(256, 384, 21)
    comp = compression.wavelet_compression(rgb)
    plain = codec.wavelet_encode(comp)
    ext = codec.wavelet_encode(comp, restarts=True)
    assert ext.byte_stream()[:15] == plain.byte_stream() and len(ext.restarts.records) == 6
    want = codec.wavelet_decode(plain)
    got, kernels = kernels_of(lambda: codec.wavelet_decode(hicimage.HicImage.from_bytes(ext.byte_stream())))
    assert "huffman_sync_kernel" not in kernels and "restart_load_kernel" in kernels
    assert all(np.array_equal(x, y) for ch in ("lum", "cr", "cb") for x, y in zip(got.as_dict[ch], want.as_dict[ch]))
    assert np.array_equal(compression.wavelet_decompression(got), orc.wavelet_decompression(orc.wavelet_compression(rgb)))


def test_file_driver_writes_and_reads_restart_records(tmp_path):
    """run.compress(restarts=True): the file's first 21 entries are what run.compress writes without them, and
    run.decompress gives the same pixels from either file."""
    import os
    import pickle
    import cv2
    from hiccup_b200 import hicimage, model, run
    rgb = orc.synthetic_image(96, 128, 61)
    src = os.path.join(tmp_path, "img.png")
    cv2.imwrite(src, rgb)
    a_dir, b_dir = os.path.join(tmp_path, "a"), os.path.join(tmp_path, "b")
    os.makedirs(a_dir)
    os.makedirs(b_dir)
    plain = run.compress(src, a_dir, model.Compression.JPEG)
    ext = run.compress(src, b_dir, model.Compression.JPEG, restarts=True)
    with open(plain, "rb") as f:
        p = pickle.load(f)
    with open(ext, "rb") as f:
        e = pickle.load(f)
    assert e[:21] == p and len(e) == 22 and hicimage.RestartP.matches(e[21])
    assert np.array_equal(run.decompress(plain), run.decompress(ext))
    many = run.compress_many([src, src], b_dir, model.Compression.JPEG, restarts=True)
    with open(many[0], "rb") as f:
        assert pickle.load(f) == e
