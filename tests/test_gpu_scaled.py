"""Scaled decode on the GPU: the 1/2- and 1/4-scale images (hic_dct_scaled: K7S, its fix-up, K8S) equal
tests/scaled_oracle.py bit for bit -- on the reference's own `.hic` bytes, odd shapes, images with many float64
re-evaluations, with and without restart records, whole batches, a 16384^2 image and through the file driver -- and
never run the full-image inverse kernels."""
import os
import pickle

import numpy as np
import pytest

from oracle import hiccup_oracle as orc
from tests import scaled_oracle as so
from tests.conftest import load_golden
from tests.reduced_helpers import GOLDENS_WITH_PIXELS, ODD, kernels_of, planes, tie_planes

pytestmark = pytest.mark.gpu

NEW_KERNELS = {"scaled_inverse_kernel", "scaled_fixup_kernel", "scaled_colour_kernel"}


@pytest.mark.parametrize("scale", [2, 4])
@pytest.mark.parametrize("name", GOLDENS_WITH_PIXELS)
def test_reference_files(name, scale):
    from hiccup_b200 import codec, hicimage
    g = load_golden(name)
    hi = hicimage.HicImage.from_bytes(pickle.loads(g["hic"].tobytes()))
    planes = {ch: g["coef_" + ch] for ch in orc.CHANNELS}
    got = codec.jpeg_scaled(hi, scale)
    want = so.jpeg_scaled(planes, scale)
    assert got.shape == want.shape and got.dtype == np.uint8
    assert np.array_equal(got, want)


@pytest.mark.parametrize("shape", ODD + [(int(h), int(w)) for h, w in np.random.default_rng(77).integers(2, 300, (6, 2))])
def test_odd_shapes_against_the_oracle(shape):
    """syn26x40, syn33x47, random sizes, and sizes whose chroma planes are one sample (or one block) wide or high."""
    from hiccup_b200 import codec, compression
    rgb = orc.synthetic_image(shape[0], shape[1], 500 + shape[0] * 7 + shape[1])
    comp = compression.jpeg_compression(rgb)
    hi = codec.jpeg_encode(comp)
    for scale in (2, 4):
        assert np.array_equal(codec.jpeg_scaled(hi, scale), so.jpeg_scaled(planes(comp), scale)), (shape, scale)


@pytest.mark.parametrize("scale", [2, 4])
def test_ties(scale, tmp_path):
    """K7S flags blocks and the fix-up changes float32 samples (scaled_stats), and the result is the oracle's."""
    from hiccup_b200 import codec, model
    from hiccup_b200.batch import DctBatchCodec
    h, w = 256, 384
    planes = tie_planes(h, w, scale, 40 + scale)
    hi = codec.jpeg_encode(model.CompressedImage(planes["lum"], planes["cr"], planes["cb"]))
    want = so.jpeg_scaled(planes, scale)
    assert np.array_equal(codec.jpeg_scaled(hi, scale), want)
    path = os.path.join(tmp_path, "t.hic")
    hi.write_file(path)
    bc = DctBatchCodec(1, h, w)
    try:
        enc = bc.read_files([path])
        assert np.array_equal(bc.decode_scaled(enc, scale)[0], want)
        st = bc.scaled_stats
        m = 8 // scale
        assert st[0] > 0 and st[1] == m * m * st[0] and st[2] > 0 and st[3] == 0, st
    finally:
        bc.close()


def test_restart_records():
    from hiccup_b200 import codec, compression, hicimage
    rgb = orc.synthetic_image(426, 640, 2100)
    comp = compression.jpeg_compression(rgb)
    plain = codec.jpeg_encode(comp)
    ext = hicimage.HicImage.from_bytes(codec.jpeg_encode(comp, restarts=True).byte_stream())
    for scale in (2, 4):
        want = so.jpeg_scaled(planes(comp), scale)
        got, k_plain = kernels_of(lambda: codec.jpeg_scaled(plain, scale))
        assert np.array_equal(got, want) and "huffman_sync_kernel" in k_plain
        got, k_ext = kernels_of(lambda: codec.jpeg_scaled(ext, scale))
        assert np.array_equal(got, want)
        assert "restart_load_kernel" in k_ext and "huffman_sync_kernel" not in k_ext


def test_kernels():
    """The scaled decode runs the entropy stage and the three scaled kernels, never K7 or K8."""
    from hiccup_b200 import codec, hicimage
    g = load_golden("lenna512")
    hi = hicimage.HicImage.from_bytes(pickle.loads(g["hic"].tobytes()))
    planes = {ch: g["coef_" + ch] for ch in orc.CHANNELS}
    for scale in (2, 4):
        got, kernels = kernels_of(lambda: codec.jpeg_scaled(hi, scale))
        assert np.array_equal(got, so.jpeg_scaled(planes, scale))
        assert NEW_KERNELS <= kernels and "expand_scatter_kernel" in kernels
        assert not kernels & {"inverse_kernel", "inverse_fixup_kernel", "upsample_colour_kernel"}


@pytest.mark.parametrize("n", [1, 3, 1024])
def test_batches(n):
    """n x 640x426: decode_scaled, its out= form and decode_scaled_device equal the single-image path image by image
    (a seeded sample of 8) and the oracle on a seeded sample of 3."""
    from hiccup_b200 import codec
    from hiccup_b200.batch import DctBatchCodec
    h, w = 426, 640
    base = np.stack([orc.synthetic_image(h, w, 2000 + i) for i in range(min(n, 16))])
    rgb = np.ascontiguousarray(base[np.arange(n) % len(base)])
    rgb[:, 0, :, 0] = (np.arange(n) // len(base)).astype(np.uint8)[:, None]        # n distinct images
    rng = np.random.default_rng(n)
    bc = DctBatchCodec(n, h, w)
    try:
        enc = bc.encode(rgb)
        his = bc.hic_images(enc)
        want = {}
        for scale in (2, 4):
            got = want[scale] = bc.decode_scaled(enc, scale).copy()
            assert got.shape == bc.scaled_shape(scale) == (n, -(-h // scale), -(-w // scale), 3)
            for i in sorted(set(rng.integers(0, n, 8).tolist()) | {0, n - 1}):
                assert np.array_equal(got[i], codec.jpeg_scaled(his[i], scale)), (scale, i)
            for i in sorted(set(rng.integers(0, n, 3).tolist())):
                planes = {ch: np.asarray(v) for ch, v in codec.jpeg_decode(his[i]).as_dict.items()}
                assert np.array_equal(got[i], so.jpeg_scaled(planes, scale)), (scale, i)
            out = np.zeros(bc.scaled_shape(scale), np.uint8)
            bc.decode_scaled(enc, scale, out=out)
            assert np.array_equal(out, got)
        bc.upload(rgb)
        bc.encode_device()
        for scale in (2, 4):
            bc.decode_scaled_device(scale)
            assert np.array_equal(bc.fetch_scaled(), want[scale])
    finally:
        bc.close()


def test_full_size_16384():
    """One 16384^2 image against the oracle applied to the coefficients the codec decodes."""
    from hiccup_b200 import codec
    from hiccup_b200.batch import DctBatchCodec
    size = 16384
    rgb = np.tile(orc.synthetic_image(2048, 2048, 4300), (8, 8, 1))
    bc = DctBatchCodec(1, size, size)
    try:
        enc = bc.encode(rgb[None])
        hi = bc.hic_images(enc)[0]              # its payloads view the codec's host buffers: used before close()
        planes = {ch: np.asarray(v) for ch, v in codec.jpeg_decode(hi).as_dict.items()}
        for scale in (2, 4):
            want = so.jpeg_scaled(planes, scale)
            assert np.array_equal(bc.decode_scaled(enc, scale)[0], want)
            assert np.array_equal(codec.jpeg_scaled(hi, scale), want)
    finally:
        bc.close()


def test_file_driver(tmp_path):
    import cv2
    from hiccup_b200 import codec, hicimage, model, run
    srcs = []
    for i, (h, w) in enumerate([(40, 41), (40, 41), (72, 96), (40, 41)]):
        p = os.path.join(tmp_path, "img%d.png" % i)
        cv2.imwrite(p, orc.synthetic_image(h, w, 170 + i))
        srcs.append(p)
    files = [run.compress(p, str(tmp_path), model.Compression.JPEG, restarts=(i == 1)) for i, p in enumerate(srcs)]
    for scale in (2, 4):
        out_dir = os.path.join(tmp_path, "s%d" % scale)
        os.makedirs(out_dir)
        many = run.decompress_many(files, save_dir=out_dir, max_batch=2, scale=scale)
        for f, r in zip(files, many):
            planes = {ch: np.asarray(v) for ch, v in codec.jpeg_decode(hicimage.HicImage.from_file(f)).as_dict.items()}
            want = so.jpeg_scaled(planes, scale)
            assert np.array_equal(r, want)
            assert np.array_equal(run.decompress(f, scale=scale), want)
            assert np.array_equal(cv2.imread(os.path.join(out_dir, os.path.basename(f) + ".s%d.png" % scale)), want)
        os.remove(os.path.join(out_dir, os.path.basename(files[2]) + ".s%d.png" % scale))
        run.main(["-d", files[2], "--scale", str(scale), "-o", out_dir])
        got = cv2.imread(os.path.join(out_dir, os.path.basename(files[2]) + ".s%d.png" % scale))
        assert np.array_equal(got, run.decompress(files[2], scale=scale))
