"""The 1/8-scale thumbnail of a DCT-mode image, defined through the oracle's own restatements of the reference
(oracle/hiccup_oracle.py: inv_dct_channel, pyr_up, ycrcb_to_rgb).  Test infrastructure: the tests compare
codec.jpeg_thumbnail and the batch thumbnails against it.

One pixel per 8x8 tile of compression.jpeg_decompression's output (out_h = 2 (h // 2), th = ceil(out_h / 8)):
  1. every block's value is what inv_dct_channel gives for it with all AC coefficients zero (a constant block);
  2. those values form Y8 (nby_l x nbx_l) and Cr16, Cb16 (nby_c x nbx_c);
  3. Cr16 and Cb16 go through pyr_up (cv2.pyrUp) to 2 nby_c x 2 nbx_c;
  4. all three are cropped to th x tw and converted by ycrcb_to_rgb.
"""
import numpy as np

from oracle import hiccup_oracle as orc


def thumbnail_shape(h, w):
    return -(-2 * (h // 2) // 8), -(-2 * (w // 2) // 8)


def dc_terms(plane):
    """The quantised DC term of every 8x8 block of a coefficient plane, (nby, nbx)."""
    plane = np.asarray(plane)
    nby, nbx = -(-plane.shape[0] // 8), -(-plane.shape[1] // 8)
    return orc.blocks_zigzag(plane)[:, 0].reshape(nby, nbx)


def dc_only_values(dc, table):
    """inv_dct_channel of the DC-only blocks, one value per block (the blocks are constant)."""
    dc = np.asarray(dc)
    nby, nbx = dc.shape
    coefs = np.zeros((8 * nby, 8 * nbx), np.float64)
    coefs[::8, ::8] = dc
    pixels = orc.inv_dct_channel(coefs, table)
    return pixels[::8, ::8]


def jpeg_thumbnail(planes):
    """planes: {"lum", "cr", "cb"} coefficient planes (what orc.jpeg_compression returns) -> (th, tw, 3) uint8."""
    h, w = np.asarray(planes["lum"]).shape
    th, tw = thumbnail_shape(h, w)
    y8 = dc_only_values(dc_terms(planes["lum"]), orc.LUM_TABLE)
    cr = orc.pyr_up(dc_only_values(dc_terms(planes["cr"]), orc.CHROMA_TABLE))
    cb = orc.pyr_up(dc_only_values(dc_terms(planes["cb"]), orc.CHROMA_TABLE))
    return orc.ycrcb_to_rgb(y8[:th, :tw], cr[:th, :tw], cb[:th, :tw])
