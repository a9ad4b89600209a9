"""Region decode at reduced scale on the GPU: a window of the 1/2- or 1/4-scale image (hic_dct_scaled_region: K7SR, its
fix-up, K8SR) or of the 1/8-scale thumbnail (hic_dct_thumbnail_region) equals the same crop of jpeg_scaled /
jpeg_thumbnail, and of the oracles, bit for bit -- on the reference's own `.hic` bytes, odd shapes, images with many
float64 re-evaluations, with and without restart records, whole batches with an origin per image and a 16384^2 image --
and never runs the whole-image transforms."""
import os
import pickle

import numpy as np
import pytest

from oracle import hiccup_oracle as orc
from tests import scaled_oracle as so
from tests import thumbnail_oracle as tho
from tests.conftest import load_golden
from tests.reduced_helpers import GOLDENS_WITH_PIXELS, ODD, fixed_windows, kernels_of, planes, tie_planes

pytestmark = pytest.mark.gpu

SCALED_KERNELS = {"scaled_region_inverse_kernel", "scaled_region_fixup_kernel", "scaled_region_colour_kernel"}
INVERSE_KERNELS = {"inverse_kernel", "inverse_fixup_kernel", "region_inverse_kernel", "scaled_inverse_kernel",
                   "scaled_region_inverse_kernel"}


def _whole(hi, scale):
    from hiccup_b200 import codec
    return codec.jpeg_thumbnail(hi) if scale == 8 else codec.jpeg_scaled(hi, scale)


def _check_windows(hi, full, scale):
    from hiccup_b200 import codec
    for top, left, rh, rw in fixed_windows(*full.shape[:2]):
        got = codec.jpeg_region(hi, top, left, rh, rw, scale=scale)
        assert got.shape == (rh, rw, 3) and got.dtype == np.uint8
        assert np.array_equal(got, full[top:top + rh, left:left + rw]), (scale, top, left, rh, rw)


@pytest.mark.parametrize("scale", [2, 4, 8])
@pytest.mark.parametrize("name", GOLDENS_WITH_PIXELS)
def test_reference_files(name, scale):
    from hiccup_b200 import hicimage
    g = load_golden(name)
    hi = hicimage.HicImage.from_bytes(pickle.loads(g["hic"].tobytes()))
    _check_windows(hi, _whole(hi, scale), scale)


@pytest.mark.parametrize("shape", ODD)
def test_odd_shapes(shape):
    """The odd shapes of the scaled tests, every scale; against the oracles themselves as well as the GPU's whole
    reduced decodes."""
    from hiccup_b200 import codec, compression
    rgb = orc.synthetic_image(shape[0], shape[1], 900 + shape[0] * 7 + shape[1])
    comp = compression.jpeg_compression(rgb)
    hi = codec.jpeg_encode(comp)
    for scale in (2, 4, 8):
        want = tho.jpeg_thumbnail(planes(comp)) if scale == 8 else so.jpeg_scaled(planes(comp), scale)
        assert np.array_equal(_whole(hi, scale), want), (shape, scale)
        _check_windows(hi, want, scale)


@pytest.mark.parametrize("scale", [2, 4])
def test_ties(scale, tmp_path):
    """A window over the first blocks of planes built so that K7S's float32 samples truncate differently: K7SR flags
    blocks, the fix-up changes samples (region_stats), no record is lost, and the result is the oracle's crop."""
    from hiccup_b200 import codec, model
    from hiccup_b200.batch import DctBatchCodec
    h, w = 256, 384
    planes = tie_planes(h, w, scale, 60 + scale)
    hi = codec.jpeg_encode(model.CompressedImage(planes["lum"], planes["cr"], planes["cb"]))
    want = so.jpeg_scaled(planes, scale)
    sh, sw = want.shape[:2]
    top, left, rh, rw = 0, 0, sh // 4 + 1, sw // 2 + 3
    assert np.array_equal(codec.jpeg_region(hi, top, left, rh, rw, scale=scale), want[:rh, :rw])
    path = os.path.join(tmp_path, "t.hic")
    hi.write_file(path)
    bc = DctBatchCodec(1, h, w)
    try:
        enc = bc.read_files([path])
        assert np.array_equal(bc.decode_regions(enc, [(top, left)], (rh, rw), scale=scale)[0], want[:rh, :rw])
        st = bc.region_stats
        assert st[0] > 0 and st[2] > 0 and st[3] == 0, st
    finally:
        bc.close()


def test_restart_records():
    from hiccup_b200 import codec, compression, hicimage
    rgb = orc.synthetic_image(426, 640, 2300)
    comp = compression.jpeg_compression(rgb)
    plain = codec.jpeg_encode(comp)
    ext = hicimage.HicImage.from_bytes(codec.jpeg_encode(comp, restarts=True).byte_stream())
    for scale, (top, left, rh, rw) in ((2, (17, 31, 112, 112)), (4, (50, 103, 56, 56)), (8, (25, 51, 28, 28))):
        full = _whole(plain, scale)
        want = full[top:top + rh, left:left + rw]
        got, k_plain = kernels_of(lambda: codec.jpeg_region(plain, top, left, rh, rw, scale=scale))
        assert np.array_equal(got, want) and "huffman_sync_kernel" in k_plain
        got, k_ext = kernels_of(lambda: codec.jpeg_region(ext, top, left, rh, rw, scale=scale))
        assert np.array_equal(got, want)
        assert "restart_load_kernel" in k_ext and "huffman_sync_kernel" not in k_ext


def test_kernels():
    """Scales 2 and 4 run the entropy stage and the three new kernels, never a whole-image transform; scale 8 runs the
    DC-only entropy stage and the 1/8-window kernel, no run-length expansion and no inverse transform at all."""
    from hiccup_b200 import codec, hicimage
    g = load_golden("lenna512")
    hi = hicimage.HicImage.from_bytes(pickle.loads(g["hic"].tobytes()))
    for scale, win in ((2, (31, 45, 112, 80)), (4, (10, 7, 56, 56)), (8, (3, 5, 28, 40))):
        full = _whole(hi, scale)
        got, kernels = kernels_of(lambda: codec.jpeg_region(hi, *win, scale=scale))
        top, left, rh, rw = win
        assert np.array_equal(got, full[top:top + rh, left:left + rw])
        if scale == 8:
            assert {"validate_dc_kernel", "thumbnail_region_kernel"} <= kernels
            assert not kernels & ({"expand_scatter_kernel", "thumbnail_kernel"} | INVERSE_KERNELS | SCALED_KERNELS)
        else:
            assert SCALED_KERNELS <= kernels and "expand_scatter_kernel" in kernels
            assert not kernels & {"inverse_kernel", "upsample_colour_kernel", "scaled_inverse_kernel", "scaled_colour_kernel",
                                  "region_inverse_kernel"}


def _origins(rng, n, sh, sw, rh, rw):
    """An origin per image: the four corners first, then random ones."""
    corners = [(0, 0), (sh - rh, sw - rw), (0, sw - rw), (sh - rh, 0)]
    o = np.stack([rng.integers(0, sh - rh + 1, n), rng.integers(0, sw - rw + 1, n)], axis=1)
    o[:min(n, 4)] = corners[:min(n, 4)]
    return o.astype(np.int32)


def _crops(full, origins, rh, rw):
    return np.stack([full[i, t:t + rh, l:l + rw] for i, (t, l) in enumerate(origins)])


@pytest.mark.parametrize("n", [1, 3, 1024])
def test_batches(n):
    """n x 640x426 with an origin per image, edge origins included: decode_regions, its out= form and
    decode_regions_device + fetch_regions equal the crops of decode_scaled / thumbnails image by image; scales and
    sizes alternate on one codec."""
    from hiccup_b200.batch import DctBatchCodec
    h, w = 426, 640
    base = np.stack([orc.synthetic_image(h, w, 2400 + i) for i in range(min(n, 16))])
    rgb = np.ascontiguousarray(base[np.arange(n) % len(base)])
    rgb[:, 0, :, 0] = (np.arange(n) // len(base)).astype(np.uint8)[:, None]        # n distinct images
    rng = np.random.default_rng(n)
    bc = DctBatchCodec(n, h, w)
    try:
        enc = bc.encode(rgb)
        full = {s: (bc.thumbnails(enc) if s == 8 else bc.decode_scaled(enc, s)).copy() for s in (2, 4, 8)}
        plan = [(2, (112, 112)), (8, (28, 28)), (4, (56, 56)), (2, (17, 33)), (8, (1, 80)), (4, (107, 1))]
        cases = []
        for scale, (rh, rw) in plan:
            sh, sw = full[scale].shape[1:3]
            origins = _origins(rng, n, sh, sw, rh, rw)
            want = _crops(full[scale], origins, rh, rw)
            got = bc.decode_regions(enc, origins, (rh, rw), scale=scale)
            assert got.shape == (n, rh, rw, 3) and np.array_equal(got, want), (scale, rh, rw)
            if scale == 8:
                assert not bc.region_stats.any()
            out = np.zeros((n, rh, rw, 3), np.uint8)
            bc.decode_regions(enc, origins, (rh, rw), out, scale)
            assert np.array_equal(out, want), (scale, rh, rw)
            cases.append((scale, rh, rw, origins, want))
        bc.upload(rgb)
        bc.encode_device()
        for scale, rh, rw, origins, want in cases:
            bc.decode_regions_device(origins, (rh, rw), scale=scale)
            assert np.array_equal(bc.fetch_regions(), want), (scale, rh, rw)
    finally:
        bc.close()


def test_full_size_16384():
    """One 16384^2 file: a 256 x 256 tile at 1/8 and at 1/2 scale equals the crop of the whole reduced decode."""
    from hiccup_b200 import codec
    from hiccup_b200.batch import DctBatchCodec
    size = 16384
    rgb = np.tile(orc.synthetic_image(2048, 2048, 4400), (8, 8, 1))
    bc = DctBatchCodec(1, size, size)
    try:
        enc = bc.encode(rgb[None])
        hi = bc.hic_images(enc)[0]              # its payloads view the codec's host buffers: used before close()
        for scale, (top, left) in ((8, (1000, 1792)), (2, (5000, 3333))):
            full = _whole(hi, scale)
            want = full[top:top + 256, left:left + 256]
            assert np.array_equal(codec.jpeg_region(hi, top, left, 256, 256, scale=scale), want)
            assert np.array_equal(bc.decode_regions(enc, [(top, left)], (256, 256), scale=scale)[0], want)
    finally:
        bc.close()
