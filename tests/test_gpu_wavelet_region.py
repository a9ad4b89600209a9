"""Wavelet region decode on the GPU: windows of the full-resolution and 1/2- to 1/2^L-scale images (hic_wavelet_region)
equal the crops they replace bit for bit -- tests/wavelet_scaled_oracle.py's image on the reference's `.hic` files and
on random flat streams whose samples wrap, the batch codec's full and scaled decodes at every level count and other
multipliers, files with restart records and C4's 7680x4320 image -- and never run the full or level-by-level inverse."""
import ctypes
import json
import pickle

import numpy as np
import pytest

from oracle import hiccup_oracle as orc
from tests import wavelet_scaled_oracle as wso
from tests.conftest import load_golden
from tests.reduced_helpers import fixed_windows, kernels_of
from tests.test_gpu_wavelet_scaled import DEFAULT, _flat_stream, _planes
from tests.test_gpu_wavelet_settings import wavelet_settings
from tests.test_wavelet_scaled_host import random_planes

pytestmark = pytest.mark.gpu

FULL_PATH = {"wavelet_inverse_kernel", "wavelet_inverse_level_kernel", "wavelet_finish_kernel",
             "wavelet_approximation_load_kernel", "wavelet_scaled_finish_kernel"}


@pytest.mark.parametrize("name", ["w_syn64", "w_syn48x80", "w_flat32", "ws_l2", "ws_l5"])
def test_reference_files(name):
    from hiccup_b200 import codec, hicimage
    g = load_golden(name)
    cfg = json.loads(str(g["settings"])) if "settings" in g else dict(DEFAULT, haar=False)
    levels = cfg["levels"]
    planes = {ch: [g["band_%s_%d" % (ch, i)] for i in range(3 * levels + 1)] for ch in orc.CHANNELS}
    hi = hicimage.HicImage.from_bytes(pickle.loads(g["hic"].tobytes()))
    with wavelet_settings(cfg, haar=cfg["haar"]):
        for k in range(levels + 1):
            want = wso.wavelet_scaled(planes, 1 << k, cfg["multiplier"])
            for top, left, rh, rw in fixed_windows(*want.shape[:2]):
                got = codec.wavelet_region(hi, top, left, rh, rw, 1 << k)
                assert got.shape == (rh, rw, 3) and got.dtype == np.uint8
                assert np.array_equal(got, want[top:top + rh, left:left + rw]), (name, k, top, left, rh, rw)


def _abi_windows(ih, iw):
    """(rh, rw, [origin of image 0, origin of image 1]) in an ih x iw image (ih, iw > 9): 1x1 at opposite corners, the
    whole image, then odd sizes with image 0's window touching the bottom and right edges and image 1's at an odd
    origin."""
    wins = [(1, 1, [(0, 0), (ih - 1, iw - 1)]), (ih, iw, [(0, 0), (0, 0)])]
    for rh, rw in ((7, 9), (ih // 2 | 1, iw // 3 | 1), (ih - 1, iw - 1)):
        wins.append((rh, rw, [(ih - rh, iw - rw), ((ih - rh) // 2 | 1, 1)]))
    return wins


def test_random_streams_through_the_c_abi():
    """A batch of two random int16 streams (cA over the whole int16 range in the second, so samples wrap), distinct
    per-image origins, at every scale of three levels: each window equals the oracle's crop."""
    from hiccup_b200 import _lib
    lib = _lib.load()
    h, w, n, L = 200, 328, 2, 3
    rng = np.random.default_rng(57)
    planes = [random_planes(h, w, L, rng, lo=-300, hi=301), random_planes(h, w, L, rng, lo=-32768, hi=32768, ca=(-32768, 32768))]
    g = _lib.wavelet_pyramid(h, w, L)
    flat = np.concatenate([_flat_stream(p, g) for p in planes])
    d_flat = _lib.scratch(flat.nbytes)
    d_flat.upload(flat)
    work = _lib.scratch(8 * n)
    params = _lib.WaveletParams()
    params.levels, params.multiplier, params.threshold, params.threshold_index = L, 1.0, 0.0, -1
    try:
        for k in range(L + 1):
            s = 1 << k
            want = [wso.wavelet_scaled(p, s) for p in planes]
            for rh, rw, origins in _abi_windows(h >> k, w >> k):
                o = np.ascontiguousarray(origins, np.int32)
                d_out = _lib.scratch(n * rh * rw * 3)
                _lib.check(lib.hic_wavelet_region(d_flat.ptr, n, h, w, ctypes.byref(params), s, o.ctypes.data, rh, rw, work.ptr,
                                                  work.nbytes, d_out.ptr, None))
                got = d_out.download(np.uint8, n * rh * rw * 3).reshape(n, rh, rw, 3)
                d_out.free()
                for i, (top, left) in enumerate(origins):
                    assert np.array_equal(got[i], want[i][top:top + rh, left:left + rw]), (s, i, top, left, rh, rw)
    finally:
        d_flat.free()
        work.free()


def test_entry_point_refuses_bad_arguments():
    from hiccup_b200 import _lib
    lib = _lib.load()
    flat, work, out = _lib.scratch(1 << 16), _lib.scratch(64), _lib.scratch(1 << 12)       # 64 x 64, three levels
    flat.zero()
    params = _lib.WaveletParams()
    params.levels, params.multiplier, params.threshold, params.threshold_index = 3, 1.0, 0.0, -1
    p = ctypes.byref(params)

    def call(h=64, w=64, s=1, origin=(0, 0), rh=8, rw=8, work_bytes=8, n=1):
        o = np.ascontiguousarray(np.tile(np.asarray(origin, np.int32), (n, 1)))
        return lib.hic_wavelet_region(flat.ptr, n, h, w, p, s, o.ctypes.data, rh, rw, work.ptr, work_bytes, out.ptr, None)
    try:
        assert call() == 0 and call(s=8, origin=(7, 7), rh=1, rw=1) == 0 and call(n=2, work_bytes=16) == 0
        _lib.sync()
        for kw in (dict(s=0), dict(s=3), dict(s=16), dict(h=60), dict(w=36), dict(rh=0), dict(rw=0), dict(origin=(-1, 0)),
                   dict(origin=(57, 0)), dict(origin=(0, 57)), dict(s=2, origin=(25, 0)), dict(work_bytes=7),
                   dict(n=2, work_bytes=15)):
            assert call(**kw) != 0, kw
    finally:
        for b in (flat, work, out):
            b.free()


def _crop(img, origins, rh, rw):
    return np.stack([img[i, t:t + rh, l:l + rw] for i, (t, l) in enumerate(origins)])


SETTINGS = [dict(levels=l, multiplier=m, threshold=5, quality_factor=1) for l in (1, 2, 3, 4, 5) for m in (2, 0.5)]


@pytest.mark.parametrize("cfg", SETTINGS, ids=lambda c: "L%d_m%g" % (c["levels"], c["multiplier"]))
def test_settings(cfg):
    """Every level count and multipliers 2 and 0.5 through WaveletBatchCodec: windows at every scale equal the crops of
    decode() (scale 1) and decode_scaled()."""
    from hiccup_b200.batch import WaveletBatchCodec
    L = cfg["levels"]
    n, h, w = 2, 64, 96
    rgb = np.stack([orc.synthetic_image(h, w, 700 + L + i) for i in range(n)])
    with wavelet_settings(cfg):
        bc = WaveletBatchCodec(n, h, w, value_bins=1 << 14)        # a 5-level cA reaches +-8192
        try:
            enc = bc.encode(rgb)
            for k in range(L + 1):
                s = 1 << k
                full = bc.decode(enc).copy() if k == 0 else bc.decode_scaled(enc, s).copy()
                ih, iw = h >> k, w >> k
                for rh, rw in {(1, 1), (ih, iw), (min(5, ih), min(7, iw)), ((ih + 1) // 2, (iw + 1) // 2 | 1)}:
                    origins = [(ih - rh, iw - rw), ((ih - rh) // 2 | (1 if ih - rh else 0), 1 if iw - rw else 0)]
                    assert np.array_equal(bc.decode_regions(enc, origins, (rh, rw), scale=s), _crop(full, origins, rh, rw)), (s, rh, rw)
        finally:
            bc.close()


@pytest.mark.parametrize("cfg", [DEFAULT, dict(levels=2, multiplier=2, threshold=3, quality_factor=0.7)],
                         ids=["defaults", "general"])
def test_batch_paths(cfg):
    """decode_regions, its out= form and decode_regions_device + fetch_regions against crops of decode / decode_scaled,
    image by image, and against codec.wavelet_region of each image's file."""
    from hiccup_b200 import codec
    from hiccup_b200.batch import WaveletBatchCodec
    n, h, w = 5, 136, 264
    rgb = np.stack([orc.synthetic_image(h, w, 900 + i) for i in range(n)])
    rng = np.random.default_rng(5)
    with wavelet_settings(cfg):
        bc = WaveletBatchCodec(n, h, w)
        try:
            enc = bc.encode(rgb)
            his = bc.hic_images(enc)
            wants = {}
            for k in range(cfg["levels"] + 1):
                s = 1 << k
                full = bc.decode(enc).copy() if k == 0 else bc.decode_scaled(enc, s).copy()
                ih, iw = h >> k, w >> k
                rh, rw = max(1, ih // 3) | 1, max(1, iw // 4) | 1
                origins = np.stack([rng.integers(0, ih - rh + 1, n), rng.integers(0, iw - rw + 1, n)], axis=1)
                want = wants[s] = (origins, rh, rw, _crop(full, origins, rh, rw))
                got = bc.decode_regions(enc, origins, (rh, rw), scale=s)
                assert got.shape == (n, rh, rw, 3) and np.array_equal(got, want[3]), s
                out = np.zeros((n, rh, rw, 3), np.uint8)
                bc.decode_regions(enc, origins, (rh, rw), out=out, scale=s)
                assert np.array_equal(out, want[3]), s
                for i in (0, n - 1):
                    t, l = (int(v) for v in origins[i])
                    assert np.array_equal(codec.wavelet_region(his[i], t, l, rh, rw, s), want[3][i]), (s, i)
            bc.upload(rgb)
            bc.encode_device()
            for s, (origins, rh, rw, want) in wants.items():
                bc.decode_regions_device(origins, (rh, rw), scale=s)
                assert np.array_equal(bc.fetch_regions(), want), s
            for bad in (3, 1 << (cfg["levels"] + 1)):
                with pytest.raises(ValueError):
                    bc.decode_regions(enc, np.zeros((n, 2), int), (1, 1), scale=bad)
            with pytest.raises(ValueError):
                bc.decode_regions(enc, np.zeros((n - 1, 2), int), (1, 1))
        finally:
            bc.close()


def test_kernels_at_the_defaults():
    """At the default settings a window at every scale is one wavelet_region_kernel launch after the entropy stage:
    neither K10 nor the level-by-level inverse runs."""
    from hiccup_b200 import codec, compression
    from hiccup_b200.batch import WaveletBatchCodec
    rgb = orc.synthetic_image(256, 384, 78)
    hi = codec.wavelet_encode(compression.wavelet_compression(rgb))
    planes = _planes(codec.wavelet_decode(hi))
    for s in (1, 2, 4, 8):
        got, kernels = kernels_of(lambda: codec.wavelet_region(hi, 3, 5, 21, 17, s))
        assert np.array_equal(got, wso.wavelet_scaled(planes, s)[3:24, 5:22]), s
        assert "wavelet_region_kernel" in kernels and "expand_scatter_kernel" in kernels
        assert not kernels & FULL_PATH, kernels & FULL_PATH
    bc = WaveletBatchCodec(2, 256, 384)
    try:
        bc.upload(np.stack([rgb, rgb[::-1].copy()]))
        bc.encode_device()
        _, kernels = kernels_of(lambda: bc.decode_regions_device([(0, 0), (1, 2)], (9, 9), scale=1))
        assert "wavelet_region_kernel" in kernels and not kernels & FULL_PATH
    finally:
        bc.close()


def test_restart_records():
    from hiccup_b200 import codec, compression, hicimage
    rgb = orc.synthetic_image(432, 640, 2300)
    comp = compression.wavelet_compression(rgb)
    plain = codec.wavelet_encode(comp)
    ext = hicimage.HicImage.from_bytes(codec.wavelet_encode(comp, restarts=True).byte_stream())
    planes = _planes(codec.wavelet_decode(plain))
    for s in (1, 2, 4, 8):
        top, left, rh, rw = 431 // s - 20, 7, 21, 640 // s - 7
        want = wso.wavelet_scaled(planes, s)[top:top + rh, left:left + rw]
        got, k_plain = kernels_of(lambda: codec.wavelet_region(plain, top, left, rh, rw, s))
        assert np.array_equal(got, want) and "huffman_sync_kernel" in k_plain
        got, k_ext = kernels_of(lambda: codec.wavelet_region(ext, top, left, rh, rw, s))
        assert np.array_equal(got, want)
        assert "restart_load_kernel" in k_ext and "huffman_sync_kernel" not in k_ext


def test_full_size_c4():
    """C4's 7680x4320 image: a 1920x1080 window at scale 1 against the crop of the device full decode, and windows at
    1/2, 1/4 and 1/8 against the oracle's crops."""
    from hiccup_b200 import codec
    from hiccup_b200.batch import WaveletBatchCodec
    h, w = 4320, 7680
    rgb = np.tile(orc.synthetic_image(1080, 1920, 4400), (4, 4, 1))
    rgb[::7, ::5] = 255 - rgb[::7, ::5]
    bc = WaveletBatchCodec(1, h, w)
    try:
        enc = bc.encode(rgb[None])
        hi = bc.hic_images(enc)[0]
        full = bc.decode(enc)[0].copy()
        top, left = 1601, 2883
        assert np.array_equal(bc.decode_regions(enc, [(top, left)], (1080, 1920))[0], full[top:top + 1080, left:left + 1920])
        assert np.array_equal(codec.wavelet_region(hi, top, left, 1080, 1920), full[top:top + 1080, left:left + 1920])
        planes = _planes(codec.wavelet_decode(hi))
        for s in (2, 4, 8):
            want = wso.wavelet_scaled(planes, s)
            top, left, rh, rw = (h // s) - 257, 1001 // s, 256, 256
            assert np.array_equal(bc.decode_regions(enc, [(top, left)], (rh, rw), scale=s)[0], want[top:top + rh, left:left + rw]), s
            assert np.array_equal(codec.wavelet_region(hi, top, left, rh, rw, s), want[top:top + rh, left:left + rw]), s
    finally:
        bc.close()
