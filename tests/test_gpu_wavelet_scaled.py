"""Wavelet scaled decode on the GPU: the 1/2- to 1/2^L-scale images (hic_wavelet_scaled_general) equal
tests/wavelet_scaled_oracle.py bit for bit -- on the reference's `.hic` files, random flat streams whose samples wrap,
every level count and other multipliers, whole batches, files with restart records and C4's 7680x4320 image -- and
never run the full inverse."""
import ctypes
import json
import os
import pickle

import numpy as np
import pytest

from oracle import hiccup_oracle as orc
from tests import wavelet_scaled_oracle as wso
from tests.conftest import load_golden
from tests.reduced_helpers import kernels_of
from tests.test_gpu_wavelet_settings import wavelet_settings
from tests.test_wavelet_scaled_host import random_planes

pytestmark = pytest.mark.gpu

DEFAULT = dict(levels=3, multiplier=1, threshold=5, quality_factor=1)


def _planes(comp):
    return {ch: [np.asarray(b) for b in v] for ch, v in comp.as_dict.items()}


@pytest.mark.parametrize("name", ["w_syn64", "w_syn48x80", "w_flat32", "ws_l2", "ws_l5"])
def test_reference_files(name):
    from hiccup_b200 import codec, hicimage
    g = load_golden(name)
    cfg = json.loads(str(g["settings"])) if "settings" in g else dict(DEFAULT, haar=False)
    levels = cfg["levels"]
    planes = {ch: [g["band_%s_%d" % (ch, i)] for i in range(3 * levels + 1)] for ch in orc.CHANNELS}
    hi = hicimage.HicImage.from_bytes(pickle.loads(g["hic"].tobytes()))
    with wavelet_settings(cfg, haar=cfg["haar"]):
        for k in range(1, levels + 1):
            got = codec.wavelet_scaled(hi, 1 << k)
            want = wso.wavelet_scaled(planes, 1 << k, cfg["multiplier"])
            assert got.shape == want.shape and got.dtype == np.uint8
            assert np.array_equal(got, want), (name, k)


def _flat_stream(planes, g):
    """The flat zigzag stream (hic_layout_flat) of one image's sub-bands, as int16."""
    chan = 64 * ((int(g.len) + 63) // 64)
    out = np.zeros(3 * chan, np.int16)
    for c, ch in enumerate(orc.CHANNELS):
        lin = np.concatenate([orc.zigzag(b) for b in planes[ch]])
        out[c * chan:c * chan + lin.size] = lin
    return out


def test_random_streams():
    """Random int16 streams of a batch of two (cA3 over the whole int16 range in the second image, so samples wrap on
    + 256) at every scale of the default settings, against the oracle."""
    from hiccup_b200 import _lib
    lib = _lib.load()
    h, w, n = 200, 328, 2
    rng = np.random.default_rng(31)
    planes = [random_planes(h, w, 3, rng, lo=-300, hi=301), random_planes(h, w, 3, rng, lo=-32768, hi=32768, ca=(-32768, 32768))]
    g = _lib.wavelet_pyramid(h, w, 3)
    flat = np.concatenate([_flat_stream(p, g) for p in planes])
    d_flat = _lib.scratch(flat.nbytes)
    d_flat.upload(flat)
    work = _lib.scratch(_lib.wavelet_work_bytes(n, h, w))
    params = _lib.WaveletParams()
    params.levels, params.multiplier, params.threshold, params.threshold_index = 3, 1.0, 0.0, -1
    try:
        for s in (2, 4, 8):
            shape = (n, h // s, w // s, 3)
            d_out = _lib.scratch(int(np.prod(shape)))
            _lib.check(lib.hic_wavelet_scaled_general(d_flat.ptr, n, h, w, ctypes.byref(params), s, work.ptr, d_out.ptr, None))
            got = d_out.download(np.uint8, int(np.prod(shape))).reshape(shape)
            d_out.free()
            for i in range(n):
                assert np.array_equal(got[i], wso.wavelet_scaled(planes[i], s)), (s, i)
    finally:
        d_flat.free()
        work.free()


def test_entry_points_refuse_bad_arguments():
    from hiccup_b200 import _lib
    lib = _lib.load()
    d = _lib.scratch(1 << 20)
    params = _lib.WaveletParams()
    params.levels, params.multiplier, params.threshold, params.threshold_index = 3, 1.0, 0.0, -1
    try:
        for s in (0, 1, 3, 16):
            assert lib.hic_wavelet_scaled_general(d.ptr, 1, 64, 64, ctypes.byref(params), s, d.ptr, d.ptr, None) != 0
        assert lib.hic_wavelet_scaled_general(d.ptr, 1, 60, 64, ctypes.byref(params), 2, d.ptr, d.ptr, None) != 0
    finally:
        d.free()


SETTINGS = [dict(levels=l, multiplier=m, threshold=5, quality_factor=1) for l in (1, 2, 3, 4, 5) for m in (2, 0.5)] + \
           [dict(levels=l, multiplier=1, threshold=3, quality_factor=1) for l in (1, 2, 4, 5)]


@pytest.mark.parametrize("cfg", SETTINGS, ids=lambda c: "L%d_m%g" % (c["levels"], c["multiplier"]))
def test_settings(cfg):
    """Every level count and multipliers 2 and 0.5 on synthetic encodes: the batch codec at every scale, and the file
    path where the reference's decoder reads the level count (2, 3, 5)."""
    from hiccup_b200 import codec, compression
    from hiccup_b200.batch import WaveletBatchCodec
    L = cfg["levels"]
    h, w = 64, 96
    rgb = np.stack([orc.synthetic_image(h, w, 600 + L + i) for i in range(2)])
    with wavelet_settings(cfg):
        bc = WaveletBatchCodec(2, h, w, value_bins=1 << 14)        # a 5-level cA reaches +-8192
        try:
            enc = bc.encode(rgb)
            for k in range(1, L + 1):
                got = bc.decode_scaled(enc, 1 << k)
                for i in range(2):
                    want = wso.wavelet_scaled(orc.wavelet_compression(rgb[i], **cfg), 1 << k, cfg["multiplier"])
                    assert np.array_equal(got[i], want), (k, i)
        finally:
            bc.close()
        if L in (2, 3, 5):
            hi = codec.wavelet_encode(compression.wavelet_compression(rgb[0]))
            planes = _planes(codec.wavelet_decode(hi))
            for k in range(1, L + 1):
                got, kernels = kernels_of(lambda: codec.wavelet_scaled(hi, 1 << k))
                assert np.array_equal(got, wso.wavelet_scaled(planes, 1 << k, cfg["multiplier"])), k
                assert "wavelet_scaled_finish_kernel" in kernels and "wavelet_finish_kernel" not in kernels


def test_kernels_at_the_defaults():
    """At the default settings the general kernels run k levels short of the full inverse, and K10 does not."""
    from hiccup_b200 import codec, compression
    rgb = orc.synthetic_image(256, 384, 77)
    hi = codec.wavelet_encode(compression.wavelet_compression(rgb))
    planes = _planes(codec.wavelet_decode(hi))
    for s in (2, 4, 8):
        got, kernels = kernels_of(lambda: codec.wavelet_scaled(hi, s))
        assert np.array_equal(got, wso.wavelet_scaled(planes, s))
        assert "wavelet_scaled_finish_kernel" in kernels and "expand_scatter_kernel" in kernels
        assert ("wavelet_inverse_level_kernel" in kernels) == (s != 8)
        assert not kernels & {"wavelet_inverse_kernel", "wavelet_finish_kernel"}


@pytest.mark.parametrize("cfg", [DEFAULT, dict(levels=2, multiplier=2, threshold=3, quality_factor=0.7)],
                         ids=["defaults", "general"])
def test_batches(cfg, tmp_path):
    from hiccup_b200 import codec
    from hiccup_b200.batch import WaveletBatchCodec
    n, h, w = 5, 136, 264
    rgb = np.stack([orc.synthetic_image(h, w, 800 + i) for i in range(n)])
    with wavelet_settings(cfg):
        bc = WaveletBatchCodec(n, h, w)
        try:
            enc = bc.encode(rgb)
            full = bc.decode(enc).copy()
            his = bc.hic_images(enc)
            paths = [os.path.join(tmp_path, "%d.hic" % i) for i in range(n)]
            bc.write_files(enc, paths)
            from_files = bc.read_files(paths)
            want = {}
            for k in range(1, cfg["levels"] + 1):
                s = 1 << k
                got = want[s] = bc.decode_scaled(enc, s).copy()
                assert got.shape == bc.scaled_shape(s) == (n, h // s, w // s, 3)
                for i in range(n):
                    assert np.array_equal(got[i], codec.wavelet_scaled(his[i], s)), (s, i)
                out = np.zeros(bc.scaled_shape(s), np.uint8)
                assert bc.decode_scaled(enc, s, out=out) is not None and np.array_equal(out, got)
                assert np.array_equal(bc.decode_scaled(from_files, s), got)
            bc.upload(rgb)
            bc.encode_device()
            for s, v in want.items():
                bc.decode_scaled_device(s)
                assert np.array_equal(bc.fetch_scaled(), v)
            assert np.array_equal(bc.decode(enc), full)
            for bad in (1, 3, 1 << (cfg["levels"] + 1)):
                with pytest.raises(ValueError):
                    bc.decode_scaled(enc, bad)
        finally:
            bc.close()


def test_restart_records():
    from hiccup_b200 import codec, compression, hicimage
    rgb = orc.synthetic_image(432, 640, 2200)
    comp = compression.wavelet_compression(rgb)
    plain = codec.wavelet_encode(comp)
    ext = hicimage.HicImage.from_bytes(codec.wavelet_encode(comp, restarts=True).byte_stream())
    planes = _planes(codec.wavelet_decode(plain))
    for s in (2, 4, 8):
        want = wso.wavelet_scaled(planes, s)
        got, k_plain = kernels_of(lambda: codec.wavelet_scaled(plain, s))
        assert np.array_equal(got, want) and "huffman_sync_kernel" in k_plain
        got, k_ext = kernels_of(lambda: codec.wavelet_scaled(ext, s))
        assert np.array_equal(got, want)
        assert "restart_load_kernel" in k_ext and "huffman_sync_kernel" not in k_ext


def test_full_size_c4():
    """C4's 7680x4320 image at every scale, whole image against the oracle on the decoded sub-bands."""
    from hiccup_b200 import codec
    from hiccup_b200.batch import WaveletBatchCodec
    h, w = 4320, 7680
    rgb = np.tile(orc.synthetic_image(1080, 1920, 4400), (4, 4, 1))
    rgb[::7, ::5] = 255 - rgb[::7, ::5]
    bc = WaveletBatchCodec(1, h, w)
    try:
        enc = bc.encode(rgb[None])
        hi = bc.hic_images(enc)[0]
        planes = _planes(codec.wavelet_decode(hi))
        for s in (2, 4, 8):
            want = wso.wavelet_scaled(planes, s)
            assert np.array_equal(bc.decode_scaled(enc, s)[0], want), s
            assert np.array_equal(codec.wavelet_scaled(hi, s), want), s
    finally:
        bc.close()
