"""Region decode on the GPU: every window (hic_dct_region: K7R, its fix-up, K8R) equals, bit for bit, the same slice
of the full decode -- of the reference's own `.hic` bytes, at every origin of small images, for odd shapes against
the oracle, with many float64 re-evaluations, with and without restart records, for whole batches, on a 16384^2
image and through the file driver -- and never runs the full-image inverse kernels."""
import os
import pickle

import numpy as np
import pytest

from oracle import hiccup_oracle as orc
from tests.conftest import load_golden
from tests.reduced_helpers import GOLDENS_WITH_PIXELS, fixed_windows, kernels_of

pytestmark = pytest.mark.gpu

NEW_KERNELS = {"region_inverse_kernel", "region_fixup_kernel", "region_colour_kernel"}


def _check_windows(hi, full):
    from hiccup_b200 import codec
    for top, left, rh, rw in fixed_windows(*full.shape[:2]):
        got = codec.jpeg_region(hi, top, left, rh, rw)
        assert got.shape == (rh, rw, 3) and got.dtype == np.uint8
        assert np.array_equal(got, full[top:top + rh, left:left + rw]), (top, left, rh, rw)


@pytest.mark.parametrize("name", GOLDENS_WITH_PIXELS)
def test_reference_files(name):
    from hiccup_b200 import codec, hicimage
    g = load_golden(name)
    hi = hicimage.HicImage.from_bytes(pickle.loads(g["hic"].tobytes()))
    _check_windows(hi, g["rgb_out"])


@pytest.mark.parametrize("name", ["tiny16", "flat32", "noise32x64", "syn48x80", "syn64"])
def test_every_origin(name):
    """Batches holding one copy of the image per valid origin: every window of each size, 1024 at a time."""
    from hiccup_b200.batch import DctBatchCodec
    g = load_golden(name)
    rgb, full = g["rgb"], g["rgb_out"]
    h, w = rgb.shape[:2]
    out_h, out_w = full.shape[:2]
    for rh, rw in sorted({(1, 1), (1, out_w), (out_h, 1), (7, 9), (16, 16), (17, 33), (9, 7), (out_h, out_w)}):
        if rh > out_h or rw > out_w:
            continue
        every = np.array([(t, l) for t in range(out_h - rh + 1) for l in range(out_w - rw + 1)], np.int32)
        for a in range(0, len(every), 1024):                # batches of up to 1024 images, one launch each
            origins = every[a:a + 1024]
            n = len(origins)
            bc = DctBatchCodec(n, h, w)
            try:
                enc = bc.encode(np.ascontiguousarray(np.broadcast_to(rgb, (n,) + rgb.shape)))
                got = bc.decode_regions(enc, origins, (rh, rw))
                assert got.shape == (n, rh, rw, 3)
                for i, (t, l) in enumerate(origins):
                    assert np.array_equal(got[i], full[t:t + rh, l:l + rw]), (rh, rw, t, l)
            finally:
                bc.close()


@pytest.mark.parametrize("shape", [(33, 47), (26, 40), (64, 106), (9, 17), (3, 5), (5, 3), (2, 2)])
def test_odd_shapes_against_the_oracle(shape):
    from hiccup_b200 import codec, compression
    rgb = orc.synthetic_image(shape[0], shape[1], 900 + shape[0] * 7 + shape[1])
    comp = compression.jpeg_compression(rgb)
    full = orc.jpeg_decompression({ch: np.asarray(v) for ch, v in comp.as_dict.items()})
    _check_windows(codec.jpeg_encode(comp), full)


def _wrapping_planes(h, w, seed):
    rng = np.random.default_rng(seed)
    planes = {}
    for ch, shape in (("lum", (h, w)), ("cr", (h // 2, w // 2)), ("cb", (h // 2, w // 2))):
        p = rng.integers(-40, 41, shape).astype(np.int32) * (rng.random(shape) < 0.5)
        p[::8, ::8] = rng.integers(-6000, 6000, p[::8, ::8].shape)
        planes[ch] = p.astype(np.int32)
    return planes


@pytest.mark.parametrize("h,w,seed", [(83, 122, 19), (64, 106, 20)])
def test_ties(h, w, seed, tmp_path):
    """Coefficients with large DC terms (samples that wrap) and dense AC terms: K7 flags many blocks.  The windows
    equal the crops, the region decode re-evaluates samples in float64, and a whole-image window flags exactly the
    blocks the full decode flags."""
    from hiccup_b200 import codec, model
    from hiccup_b200.batch import DctBatchCodec
    planes = _wrapping_planes(h, w, seed)
    hi = codec.jpeg_encode(model.CompressedImage(planes["lum"], planes["cr"], planes["cb"]))
    full = orc.jpeg_decompression(planes)
    path = os.path.join(tmp_path, "t.hic")
    hi.write_file(path)
    bc = DctBatchCodec(1, h, w)
    try:
        enc = bc.read_files([path])
        assert np.array_equal(bc.decode(enc)[0], full)
        flagged = int(bc.inverse_stats[0])
        assert flagged > 0 and int(bc.inverse_stats[1]) > 0
        out_h, out_w = full.shape[:2]
        whole = bc.decode_regions(enc, [(0, 0)], (out_h, out_w))
        assert np.array_equal(whole[0], full)
        assert int(bc.region_stats[0]) == flagged and int(bc.region_stats[1]) == int(bc.inverse_stats[1])
        assert int(bc.region_stats[3]) == 0
        seen = 0
        for top, left, rh, rw in fixed_windows(out_h, out_w):
            got = bc.decode_regions(enc, [(top, left)], (rh, rw))
            assert np.array_equal(got[0], full[top:top + rh, left:left + rw]), (top, left, rh, rw)
            assert int(bc.region_stats[0]) <= flagged
            seen += int(bc.region_stats[1])
        assert seen > 0
    finally:
        bc.close()


def test_restart_records():
    from hiccup_b200 import codec, compression, hicimage
    rgb = orc.synthetic_image(426, 640, 2100)
    comp = compression.jpeg_compression(rgb)
    full = compression.jpeg_decompression(comp)
    plain = codec.jpeg_encode(comp)
    ext = hicimage.HicImage.from_bytes(codec.jpeg_encode(comp, restarts=True).byte_stream())
    for top, left, rh, rw in [(37, 101, 224, 224), (0, 0, 426, 640), (425, 639, 1, 1)]:
        want = full[top:top + rh, left:left + rw]
        got, k_plain = kernels_of(lambda: codec.jpeg_region(plain, top, left, rh, rw))
        assert np.array_equal(got, want) and "huffman_sync_kernel" in k_plain
        got, k_ext = kernels_of(lambda: codec.jpeg_region(ext, top, left, rh, rw))
        assert np.array_equal(got, want)
        assert "restart_load_kernel" in k_ext and "huffman_sync_kernel" not in k_ext


def test_kernels():
    """The region decode runs the entropy stage and the three region kernels, never K7 or K8 over the whole image."""
    from hiccup_b200 import codec, hicimage
    g = load_golden("lenna512")
    hi = hicimage.HicImage.from_bytes(pickle.loads(g["hic"].tobytes()))
    got, kernels = kernels_of(lambda: codec.jpeg_region(hi, 100, 203, 64, 77))
    assert np.array_equal(got, g["rgb_out"][100:164, 203:280])
    assert NEW_KERNELS <= kernels and "expand_scatter_kernel" in kernels
    assert not kernels & {"inverse_kernel", "inverse_fixup_kernel", "upsample_colour_kernel"}


def test_c2_batch():
    """1024 x 640x426 with seeded per-image origins and 224 x 224 windows: decode_regions and decode_regions_device
    equal decode() cropped image by image."""
    from hiccup_b200.batch import DctBatchCodec
    n, h, w, rh, rw = 1024, 426, 640, 224, 224
    base = np.stack([orc.synthetic_image(h, w, 2000 + i) for i in range(16)])
    rgb = np.ascontiguousarray(base[np.arange(n) % 16])
    rgb[:, 0, :, 0] = (np.arange(n) // 16).astype(np.uint8)[:, None]        # 1024 distinct images
    rng = np.random.default_rng(224)
    origins = np.stack([rng.integers(0, h - rh + 1, n), rng.integers(0, w - rw + 1, n)], 1).astype(np.int32)
    origins[:4] = [(0, 0), (h - rh, w - rw), (0, w - rw), (h - rh, 0)]
    bc = DctBatchCodec(n, h, w)
    try:
        enc = bc.encode(rgb)
        full = bc.decode(enc).copy()
        want = np.stack([full[i, t:t + rh, l:l + rw] for i, (t, l) in enumerate(origins)])
        got = bc.decode_regions(enc, origins, (rh, rw))
        assert np.array_equal(got, want)
        out = np.zeros((n, rh, rw, 3), np.uint8)
        bc.decode_regions(enc, origins, (rh, rw), out=out)
        assert np.array_equal(out, want)
        bc.upload(rgb)
        bc.encode_device()
        bc.decode_regions_device(origins, (rh, rw))
        assert np.array_equal(bc.fetch_regions(), want)
        with pytest.raises(ValueError):
            bc.decode_regions(enc, origins[:-1], (rh, rw))                    # one origin per image
    finally:
        bc.close()


def test_full_size_16384():
    """One 16384^2 image: a 2048^2 window at an unaligned origin equals the same window of the full decode, through
    the batch codec and through the single-image function."""
    from hiccup_b200 import codec
    from hiccup_b200.batch import DctBatchCodec
    size, win, top, left = 16384, 2048, 5003, 7777
    rgb = np.tile(orc.synthetic_image(2048, 2048, 4300), (8, 8, 1))
    bc = DctBatchCodec(1, size, size)
    try:
        enc = bc.encode(rgb[None])
        want = bc.decode(enc)[0, top:top + win, left:left + win].copy()
        assert np.array_equal(bc.decode_regions(enc, [(top, left)], (win, win))[0], want)
        hi = bc.hic_images(enc)[0]              # its payloads view the codec's host buffers: used before close()
        assert np.array_equal(codec.jpeg_region(hi, top, left, win, win), want)
    finally:
        bc.close()


def test_file_driver(tmp_path):
    import cv2
    from hiccup_b200 import model, run
    srcs = []
    for i, (h, w) in enumerate([(40, 41), (40, 41), (72, 96), (40, 41)]):
        p = os.path.join(tmp_path, "img%d.png" % i)
        cv2.imwrite(p, orc.synthetic_image(h, w, 170 + i))
        srcs.append(p)
    files = [run.compress(p, str(tmp_path), model.Compression.JPEG, restarts=(i == 1)) for i, p in enumerate(srcs)]
    out_dir = os.path.join(tmp_path, "regions")
    os.makedirs(out_dir)
    region = (3, 5, 30, 31)
    many = run.decompress_many(files, save_dir=out_dir, max_batch=2, region=region)
    for f, r in zip(files, many):
        full = run.decompress(f)
        want = full[3:33, 5:36]
        assert np.array_equal(r, want)
        assert np.array_equal(run.decompress(f, region=region), want)
        assert np.array_equal(cv2.imread(os.path.join(out_dir, os.path.basename(f) + ".region.png")), want)
    os.remove(os.path.join(out_dir, os.path.basename(files[2]) + ".region.png"))
    run.main(["-d", files[2], "--region", "40,60,32,36", "-o", out_dir])
    got = cv2.imread(os.path.join(out_dir, os.path.basename(files[2]) + ".region.png"))
    assert np.array_equal(got, run.decompress(files[2])[40:72, 60:96])
