"""The wavelet scaled decode without a device: its definition (tests/wavelet_scaled_oracle.py) against the full
decode and the tile-mean property, its shapes, and the argument checks of _lib.wavelet_scale_arg and
codec.wavelet_scaled, which all come before any device work."""
import pickle

import numpy as np
import pytest

from oracle import hiccup_oracle as orc
from tests import wavelet_scaled_oracle as wso
from tests.conftest import load_golden


def random_planes(h, w, levels, rng, lo=-40, hi=41, ca=(-3000, 3001)):
    """{lum, cr, cb: 3 L + 1 int32 sub-bands} of an h x w image (h, w multiples of 2^L); cA_L in `ca`, details in
    [lo, hi)."""
    planes = {}
    for ch in orc.CHANNELS:
        bands = [rng.integers(ca[0], ca[1], (h >> levels, w >> levels)).astype(np.int32)]
        for l in range(levels, 0, -1):
            bands += [rng.integers(lo, hi, (h >> l, w >> l)).astype(np.int32) for _ in range(3)]
        planes[ch] = bands
    return planes


def tile_mean(a, s):
    return a.reshape(a.shape[0] // s, s, a.shape[1] // s, s).mean(axis=(1, 3))


@pytest.mark.parametrize("levels,shape", [(2, (64, 64)), (3, (48, 80)), (3, (64, 96)), (5, (64, 96)), (1, (6, 10))])
def test_scale_one_is_the_full_decode(levels, shape):
    rng = np.random.default_rng(levels * 100 + shape[1])
    for multiplier in (1, 2, 0.5):
        planes = random_planes(shape[0], shape[1], levels, rng)
        assert np.array_equal(wso.wavelet_scaled(planes, 1, multiplier), orc.wavelet_decompression(planes, multiplier))


@pytest.mark.parametrize("levels,shape", [(2, (64, 64)), (3, (48, 80)), (3, (64, 96)), (5, (64, 96)), (4, (32, 48))])
def test_approximation_is_the_tile_mean(levels, shape):
    """A_k * 2^-k equals the mean of each 2^k x 2^k tile of the unrounded waverec2 (floating-point noise only)."""
    rng = np.random.default_rng(levels + shape[0])
    planes = random_planes(shape[0], shape[1], levels, rng, lo=-500, hi=501)
    for multiplier in (1, 2):
        for ch in orc.CHANNELS:
            full = wso.approximation(planes[ch], 0, multiplier)
            for k in range(1, levels + 1):
                got = wso.approximation(planes[ch], k, multiplier)
                assert got.shape == (shape[0] >> k, shape[1] >> k)
                assert np.abs(got - tile_mean(full, 1 << k)).max() < 1e-9, (ch, k)


def test_approximation_at_k_equal_levels_is_ca():
    rng = np.random.default_rng(3)
    planes = random_planes(32, 64, 3, rng)
    a = wso.approximation(planes["lum"], 3)
    assert np.array_equal(a, planes["lum"][0] / 8.0)


@pytest.mark.parametrize("levels", [1, 2, 3, 4, 5])
def test_shapes(levels):
    rng = np.random.default_rng(levels)
    h, w = 3 << levels, 5 << levels
    planes = random_planes(h, w, levels, rng)
    for k in range(0, levels + 1):
        out = wso.wavelet_scaled(planes, 1 << k)
        assert out.shape == (h >> k, w >> k, 3) and out.dtype == np.uint8


def test_samples_wrap_like_the_full_decode():
    """A large cA gives samples past 255 before the cast: they wrap, as the full decode's + 256, astype(uint8) does."""
    bands = [np.full((1, 1), 2000, np.int32)] + [np.zeros((1, 1), np.int32)] * 3
    a = wso.approximation(bands, 1)
    assert a[0, 0] == 1000.0
    assert wso.scaled_channel(bands, 1)[0, 0] == (1000 + 256) & 0xFF
    assert wso.scaled_channel(bands, 0)[0, 0] == (1000 + 256) & 0xFF


def test_scale_arg():
    from hiccup_b200 import _lib
    for levels in range(1, 6):
        for k in range(1, levels + 1):
            assert _lib.wavelet_scale_arg(1 << k, levels) == k
            assert _lib.wavelet_scale_arg(np.int64(1 << k), levels) == k
        for bad in (1, 0, -2, 3, 6, 1 << (levels + 1), 2.0, True, False, None, "2"):
            with pytest.raises(ValueError):
                _lib.wavelet_scale_arg(bad, levels)


def _hic(name):
    from hiccup_b200 import hicimage
    return hicimage.HicImage.from_bytes(pickle.loads(load_golden(name)["hic"].tobytes()))


def test_codec_refusals_before_any_device_work():
    from hiccup_b200 import codec
    with pytest.raises(NotImplementedError):
        codec.wavelet_scaled(_hic("syn64"), 2)
    hi = _hic("w_syn64")
    for bad in (1, 3, 16, 2.0, True):
        with pytest.raises(ValueError):
            codec.wavelet_scaled(hi, bad)
    with pytest.raises(ValueError):
        codec.wavelet_scaled(_hic("ws_l4"), 2)          # four levels: pyramid_of_file refuses the file


def test_new_symbol_is_bound():
    from hiccup_b200 import _lib
    assert "hic_wavelet_scaled_general" in _lib.SIGNATURES and hasattr(_lib.load(), "hic_wavelet_scaled_general")
