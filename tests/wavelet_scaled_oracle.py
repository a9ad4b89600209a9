"""The wavelet scaled decode, written down (it has no counterpart in the reference).  TEST INFRASTRUCTURE ONLY.

A wavelet file of L levels holds an h x w image with h and w multiples of 2^L.  Its 1/s image, s = 2^k with
1 <= k <= L, is (h / s) x (w / s) x 3, per channel:

  1. dequantise as compression.wavelet_decompression does: A_L = cA_L as float64; detail group i (0 = coarsest,
     level L - i) times multiplier * (i*i + 1);
  2. A_k = the running approximation after the first L - k reconstruction levels of waverec2 -- waverec2 applied to
     the truncated coefficient list, so bit for bit the intermediate the full inverse holds at that point;
  3. sample = astype(uint8)(A_k * 2^-k + 256): the product is exact, the cast the full decode's;
  4. ycrcb_to_rgb of the three reduced planes (no chroma subsampling: no crop, no pyrUp).

For db1, A_k * 2^-k is the mean of each s x s tile of the unrounded full reconstruction.  At k = 0 the steps are
the full decode's.
"""
import numpy as np

from oracle import hiccup_oracle as orc
from oracle import pywt_standin as pywt


def approximation(bands, k, multiplier=None):
    """A_k * 2^-k of one channel's 3 L + 1 sub-bands, before the cast (float64)."""
    multiplier = orc.WAVELET_MULTIPLIER if multiplier is None else multiplier
    bands = [np.asarray(b) for b in bands]
    levels = (len(bands) - 1) // 3
    assert 0 <= k <= levels
    coeffs = [orc.np_round_i32(bands[0])]
    rest = bands[1:]
    for i in range(levels - k):
        coeffs.append(tuple(np.multiply(b, multiplier * (i * i + 1)) for b in rest[3 * i:3 * i + 3]))
    return np.multiply(pywt.waverec2(coeffs, "db1"), 2.0 ** -k)


def scaled_channel(bands, k, multiplier=None):
    return orc.astype_u8(np.add(approximation(bands, k, multiplier), 256))


def wavelet_scaled(planes, scale, multiplier=None):
    """The 1/scale image of a channel dict {lum, cr, cb: [3 L + 1 sub-bands]}; scale = 2^k, 0 <= k <= L."""
    k = int(scale).bit_length() - 1
    assert scale == 1 << k
    y, cr, cb = (scaled_channel(planes[c], k, multiplier) for c in orc.CHANNELS)
    return orc.ycrcb_to_rgb(y, cr, cb)
