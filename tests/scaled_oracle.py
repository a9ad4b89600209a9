"""The 1/2- and 1/4-scale images of a DCT-mode image, defined through the oracle's own restatements of the reference
(oracle/hiccup_oracle.py: pyr_up, ycrcb_to_rgb, astype_u8).  Test infrastructure: the tests compare
codec.jpeg_scaled and the batch scaled decode against it.

Scale s, m = 8 / s samples per block side:
  1. B_s is m x m: B_s[k][0] = 1, B_s[k][n] = 2 D_s(n) cos(pi n (2k+1) / (2m)), D_s(n) = sin(pi n s / 16) /
     (s sin(pi n / 16)).  For a block with coefficients only at u, v < m, B_s X B_s^T is the mean of each s x s tile
     of the unrounded 8 x 8 IDCT.  BASIS holds the correctly rounded float64 values, the bits csrc/hic_core.cuh
     commits (tests/test_scaled_host.py checks both).
  2. every block of the zero-padded plane: X = q T for u, v < m (float64, exact), A[u][k] = sum_v B[k][v] X[u][v]
     (rows first), Y[j][k] = sum_u B[j][u] A[u][k], each sum left to right from its first product, every product and
     sum rounded; sample = astype_u8(Y / 256 + 128);
  3. the samples form Y_s ((nby_l m) x (nbx_l m)) and Cr_s, Cb_s ((nby_c m) x (nbx_c m)); Cr_s and Cb_s go
     through pyr_up; all three are cropped to (ceil(out_h / s), ceil(out_w / s)), out_h = 2 (h // 2), and converted
     by ycrcb_to_rgb.
At m = 1 (B = [[1]]) this is thumbnail_oracle.jpeg_thumbnail.
"""
import numpy as np

from oracle import hiccup_oracle as orc

_B4 = ["0x1.0p+0", "0x1.cfefefc82ff2ap+0", "0x1.4e7ae9144f0fcp+0", "0x1.45d3819f43820p-1",
       "0x1.0p+0", "0x1.8056948c8d24bp-1", "-0x1.4e7ae9144f0fcp+0", "-0x1.894e984d2e2bcp+0",
       "0x1.0p+0", "-0x1.8056948c8d24bp-1", "-0x1.4e7ae9144f0fcp+0", "0x1.894e984d2e2bcp+0",
       "0x1.0p+0", "-0x1.cfefefc82ff2ap+0", "0x1.4e7ae9144f0fcp+0", "-0x1.45d3819f43820p-1"]
_B2 = ["0x1.0p+0", "0x1.480d9d073b428p+0", "0x1.0p+0", "-0x1.480d9d073b428p+0"]
BASIS = {4: np.array([float.fromhex(v) for v in _B4]).reshape(4, 4),
         2: np.array([float.fromhex(v) for v in _B2]).reshape(2, 2),
         1: np.ones((1, 1))}


def closed_form_basis(scale):
    """B_s from its closed form, evaluated with 100 significant digits (mpmath) and rounded once to float64."""
    import mpmath
    m = 8 // scale
    with mpmath.workdps(100):
        def entry(k, n):
            if n == 0:
                return mpmath.mpf(1)
            d = mpmath.sin(mpmath.pi * n * scale / 16) / (scale * mpmath.sin(mpmath.pi * n / 16))
            return 2 * d * mpmath.cos(mpmath.pi * n * (2 * k + 1) / (2 * m))
        return np.array([[float(entry(k, n)) for n in range(m)] for k in range(m)])


def scaled_shape(h, w, scale):
    return -(-2 * (h // 2) // scale), -(-2 * (w // 2) // scale)


def block_values(blocks, table, m):
    """blocks: (N, >= m, >= m) quantised coefficients (natural order) -> (N, m, m) float64 Y / 256 + 128 before the cast."""
    b = BASIS[m]
    x = (np.asarray(blocks)[:, :m, :m].astype(np.int64) * np.asarray(table)[:m, :m].astype(np.int64)).astype(np.float64)
    a = np.empty(x.shape[:1] + (m, m))
    for u in range(m):
        for k in range(m):
            acc = b[k, 0] * x[:, u, 0]
            for v in range(1, m):
                acc = acc + b[k, v] * x[:, u, v]
            a[:, u, k] = acc
    y = np.empty_like(a)
    for j in range(m):
        for k in range(m):
            acc = b[j, 0] * a[:, 0, k]
            for u in range(1, m):
                acc = acc + b[j, u] * a[:, u, k]
            y[:, j, k] = acc
    return np.add(np.divide(y, 256), 128)


def scaled_plane(plane, table, m):
    """A coefficient plane -> its reduced sample plane ((nby m) x (nbx m) uint8, whole block grid)."""
    padded = orc.pad_matrix(np.asarray(plane))
    nby, nbx = padded.shape[0] // 8, padded.shape[1] // 8
    corners = padded.reshape(nby, 8, nbx, 8)[:, :m, :, :m].swapaxes(1, 2).reshape(-1, m, m)     # only u, v < m are read
    samples = orc.astype_u8(block_values(corners, table, m))
    return samples.reshape(nby, nbx, m, m).swapaxes(1, 2).reshape(nby * m, nbx * m)


def jpeg_scaled(planes, scale):
    """planes: {"lum", "cr", "cb"} coefficient planes (what orc.jpeg_compression returns) -> (sh, sw, 3) uint8."""
    m = 8 // scale
    h, w = np.asarray(planes["lum"]).shape
    sh, sw = scaled_shape(h, w, scale)
    y = scaled_plane(planes["lum"], orc.LUM_TABLE, m)
    cr = orc.pyr_up(scaled_plane(planes["cr"], orc.CHROMA_TABLE, m))
    cb = orc.pyr_up(scaled_plane(planes["cb"], orc.CHROMA_TABLE, m))
    return orc.ycrcb_to_rgb(y[:sh, :sw], cr[:sh, :sw], cb[:sh, :sw])
