"""The wavelet region decode without a device: a window computed from the dyadic parent rectangles alone equals the crop
of tests/wavelet_scaled_oracle.py's image (at scale 1 the full decode), and every argument check of
_lib.wavelet_region_origins, codec.wavelet_region and WaveletBatchCodec's windows comes before any device work."""
import pickle

import numpy as np
import pytest

from oracle import hiccup_oracle as orc
from oracle import pywt_standin as pywt
from tests import wavelet_scaled_oracle as wso
from tests.conftest import load_golden
from tests.reduced_helpers import random_windows
from tests.test_wavelet_scaled_host import random_planes


def window_from_parents(planes, scale, top, left, rh, rw, multiplier=1):
    """The rh x rw window at (top, left) of the 1/scale image from, at each level l > k (scale = 2^k), the rows
    [top >> (l-k), (top+rh-1) >> (l-k)] and the same columns of the level's bands only, with the oracle's operations."""
    k = int(scale).bit_length() - 1
    out = []
    for ch in orc.CHANNELS:
        bands = planes[ch]
        levels = (len(bands) - 1) // 3

        def rect(l):
            s = l - k
            return top >> s, ((top + rh - 1) >> s) + 1, left >> s, ((left + rw - 1) >> s) + 1
        y0, y1, x0, x1 = rect(levels)
        a = np.asarray(orc.np_round_i32(bands[0])[y0:y1, x0:x1], np.float64)
        for i in range(levels - k):
            d = tuple(np.multiply(b[y0:y1, x0:x1], multiplier * (i * i + 1)) for b in bands[1 + 3 * i:4 + 3 * i])
            a = pywt.idwt2((a, d), "db1")                      # rows [2 y0, 2 y1) of level l - 1
            ny0, ny1, nx0, nx1 = rect(levels - i - 1)
            a = a[ny0 - 2 * y0:ny1 - 2 * y0, nx0 - 2 * x0:nx1 - 2 * x0]
            y0, y1, x0, x1 = ny0, ny1, nx0, nx1
        assert a.shape == (rh, rw)
        out.append(orc.astype_u8(np.add(np.multiply(a, 2.0 ** -k), 256)))
    return orc.ycrcb_to_rgb(*out)


@pytest.mark.parametrize("levels", [1, 2, 3, 4, 5])
def test_parent_rectangles_give_the_crop(levels):
    """Random planes whose samples wrap (cA over the whole int16 range, large details), every scale, odd origins and
    sizes: the window from the parent rectangles equals the crop of the 1/scale image, bit for bit."""
    rng = np.random.default_rng(40 + levels)
    h, w = 3 << levels, 5 << levels
    planes = random_planes(h, w, levels, rng, lo=-2000, hi=2001, ca=(-32768, 32768))
    for multiplier in (1, 0.5):
        for k in range(levels + 1):
            full = wso.wavelet_scaled(planes, 1 << k, multiplier)
            for top, left, rh, rw in random_windows(h >> k, w >> k, rng):
                got = window_from_parents(planes, 1 << k, top, left, rh, rw, multiplier)
                assert np.array_equal(got, full[top:top + rh, left:left + rw]), (k, top, left, rh, rw)


def test_origins():
    from hiccup_b200 import _lib
    for levels in range(1, 6):
        h, w = 3 << levels, 5 << levels
        for k in range(levels + 1):
            ih, iw = h >> k, w >> k
            o = _lib.wavelet_region_origins(h, w, levels, [(ih - 1, iw - 1), (0, 0)], (1, 1), 1 << k)
            assert o.dtype == np.int32 and o.shape == (2, 2) and o.flags.c_contiguous
            assert o.tolist() == [[ih - 1, iw - 1], [0, 0]]
            _lib.wavelet_region_origins(h, w, levels, [(0, 0)], (ih, iw), np.int64(1 << k))
            for origin, size in (((0, 0), (0, 1)), ((0, 0), (1, 0)), ((-1, 0), (1, 1)), ((0, -1), (1, 1)),
                                 ((1, 0), (ih, 1)), ((0, 1), (1, iw)), ((ih, 0), (1, 1)), ((0, iw), (1, 1))):
                with pytest.raises(ValueError):
                    _lib.wavelet_region_origins(h, w, levels, [origin], size, 1 << k)
        for bad in (0, 3, 1 << (levels + 1), 2.0, "4", True, None, -2):
            with pytest.raises(ValueError):
                _lib.wavelet_region_origins(h, w, levels, [(0, 0)], (1, 1), bad)
    with pytest.raises(ValueError):
        _lib.wavelet_region_origins(60, 64, 3, [(0, 0)], (1, 1), 1)           # sides must be multiples of 2^levels
    for bad in (np.zeros((0, 2), int), np.zeros((2, 3), int), np.zeros(2, int), np.zeros((1, 2))):
        with pytest.raises(ValueError):
            _lib.wavelet_region_origins(64, 64, 3, bad, (1, 1), 1)


def test_region_origins_of_dct_files_unchanged():
    """region_origins shares the bounds check; its DCT scales and messages stay as they were."""
    from hiccup_b200 import _lib
    with pytest.raises(ValueError, match=r"region 1x1 at \(26, 0\) is not inside the 26x40 decoded image"):
        _lib.region_origins(26, 40, [(26, 0)], (1, 1))
    with pytest.raises(ValueError, match=r"is not inside the 4x5 1/8-scale image"):
        _lib.region_origins(26, 40, [(4, 0)], (1, 1), 8)
    with pytest.raises(ValueError):
        _lib.region_origins(26, 40, [(0, 0)], (1, 1), 16)


def _hic(name):
    from hiccup_b200 import hicimage
    return hicimage.HicImage.from_bytes(pickle.loads(load_golden(name)["hic"].tobytes()))


def test_codec_refusals_before_any_device_work():
    """Without a device any device work would raise HicError: these raise their own errors first."""
    from hiccup_b200 import codec
    with pytest.raises(NotImplementedError):
        codec.wavelet_region(_hic("syn64"), 0, 0, 8, 8)
    hi = _hic("w_syn64")                                    # 64 x 64, three levels
    for bad in (0, 3, 16, 2.0, "4", True):
        with pytest.raises(ValueError):
            codec.wavelet_region(hi, 0, 0, 1, 1, bad)
    for top, left, rh, rw, s in ((0, 0, 0, 8, 1), (0, 0, 8, 0, 1), (-1, 0, 8, 8, 1), (0, -1, 8, 8, 1), (57, 0, 8, 8, 1),
                                 (0, 57, 8, 8, 1), (0, 0, 65, 1, 1), (25, 0, 8, 8, 2), (0, 1, 1, 8, 8)):
        with pytest.raises(ValueError):
            codec.wavelet_region(hi, top, left, rh, rw, s)
    with pytest.raises(ValueError):
        codec.wavelet_region(_hic("ws_l4"), 0, 0, 8, 8)    # four levels: pyramid_of_file refuses the file


def test_batch_origin_count_is_checked_on_the_host():
    from hiccup_b200 import _lib
    from hiccup_b200.batch import WaveletBatchCodec
    bc = WaveletBatchCodec.__new__(WaveletBatchCodec)       # no device: only the fields the checks read
    bc.n, bc.h, bc.w = 2, 64, 96
    bc.params = _lib.WaveletParams()
    bc.params.levels = 3
    for origins in (np.zeros((3, 2), int), np.zeros((1, 2), int)):
        with pytest.raises(ValueError, match="origins for a batch of 2 images"):
            bc.decode_regions_device(origins, (8, 8))
    with pytest.raises(ValueError):
        bc.decode_regions_device(np.zeros((2, 2), int), (8, 8), scale=16)
    with pytest.raises(ValueError):
        bc.decode_regions_device(np.array([[0, 0], [57, 0]]), (8, 8))


def test_new_symbol_is_bound():
    from hiccup_b200 import _lib
    assert "hic_wavelet_region" in _lib.SIGNATURES and hasattr(_lib.load(), "hic_wavelet_region")
