"""Region decode at reduced scale, the parts that need no GPU: the block selection at m = 8 / scale samples per block
against a brute-force enumeration of every tap of every output pixel, the work and tie sizes against the layout, and
the argument checks of every new entry point (they all refuse before any device work, so they run here)."""
import numpy as np
import pytest

from tests.reduced_helpers import random_windows, write_goldens

SHAPES = [(2, 2), (3, 5), (5, 3), (17, 2), (2, 17), (9, 17), (26, 40), (33, 47), (64, 81), (426, 640)] + \
    [(int(h), int(w)) for h, w in np.random.default_rng(5).integers(2, 400, (8, 2))]


def _reduced(g, scale):
    """(sh, sw) of the 1/scale image and the sample counts of its reduced planes: (luminance rows, columns), (chroma
    rows, columns)."""
    m = 8 // scale
    return (-(-g.out_h // scale), -(-g.out_w // scale)), (m * g.nby_l, m * g.nbx_l), (m * g.nby_c, m * g.nbx_c)


def _taps(first, count, n_c):
    """Reduced luminance rows and chroma rows K8SR reads for output rows [first, first + count) (columns alike): every
    pixel's own luminance row and its three pyrUp taps, chosen as K8S chooses them in the whole chroma plane."""
    o = np.arange(first, first + count)
    cy = o >> 1
    ym = np.where(cy > 0, cy - 1, 1 if n_c > 1 else 0)
    yn = np.minimum(cy + 1, n_c - 1)
    return o, np.unique(np.concatenate([ym, cy, yn]))


def _check_cover(g, scale, top, left, rh, rw, lum_rect, c_rect):
    m = 8 // scale
    (sh, sw), (nyl, nxl), (nyc, nxc) = _reduced(g, scale)
    rows_l, rows_c = _taps(top, rh, nyc)
    cols_l, cols_c = _taps(left, rw, nxc)
    by, bx, nby, nbx = lum_rect
    assert 0 <= by and by + nby <= g.nby_l and 0 <= bx and bx + nbx <= g.nbx_l
    assert rows_l.max() < nyl and cols_l.max() < nxl
    assert (rows_l // m >= by).all() and (rows_l // m < by + nby).all()
    assert (cols_l // m >= bx).all() and (cols_l // m < bx + nbx).all()
    by, bx, nby, nbx = c_rect
    assert 0 <= by and by + nby <= g.nby_c and 0 <= bx and bx + nbx <= g.nbx_c
    assert rows_c.min() >= 0 and rows_c.max() < nyc and cols_c.min() >= 0 and cols_c.max() < nxc
    assert (rows_c // m >= by).all() and (rows_c // m < by + nby).all()
    assert (cols_c // m >= bx).all() and (cols_c // m < bx + nbx).all()


@pytest.mark.parametrize("scale", [2, 4])
@pytest.mark.parametrize("h,w", SHAPES)
def test_selection_covers_every_tap(h, w, scale):
    """Corners, edges, rows, columns, the whole image and random windows of the 1/scale image; every 1 x 1 window of the
    small ones.  The rectangles lie inside the block grids, cover every sample read, and have one size per window
    size."""
    from hiccup_b200 import _lib
    g = _lib.geometry(h, w)
    (sh, sw), _, _ = _reduced(g, scale)
    assert (sh, sw) == _lib.scaled_shape(h, w, scale)
    windows = list(random_windows(sh, sw, np.random.default_rng(h * 1000 + w + scale)))
    if sh * sw <= 400:
        windows += [(t, l, 1, 1) for t in range(sh) for l in range(sw)]
    shapes = {}
    for top, left, rh, rw in windows:
        lum_rect, c_rect = _lib.scaled_region_blocks(h, w, scale, top, left, rh, rw)
        _check_cover(g, scale, top, left, rh, rw, lum_rect, c_rect)
        shapes.setdefault((rh, rw), set()).add(lum_rect[2:] + c_rect[2:])
    assert all(len(v) == 1 for v in shapes.values()), shapes


@pytest.mark.parametrize("scale", [2, 4])
@pytest.mark.parametrize("h,w", [(2, 2), (3, 5), (17, 2), (26, 40), (33, 47), (64, 81)])
def test_every_origin_of_every_size(h, w, scale):
    """Every window of every size (a spread of sizes in the larger images): covered, one rectangle size per window
    size, never fewer blocks than the worst origin needs and at most one more per axis; the sizes count those blocks."""
    from hiccup_b200 import _lib
    g = _lib.geometry(h, w)
    m = 8 // scale
    (sh, sw), _, (nyc, nxc) = _reduced(g, scale)
    pick = lambda n: range(1, n + 1) if n <= 12 else sorted({1, 2, 3, m - 1, m, m + 1, 2 * m + 1, n // 2, n - 1, n} - {0})
    for rh in pick(sh):
        for rw in pick(sw):
            shapes, need = set(), [0, 0, 0, 0]
            for top in range(sh - rh + 1):
                for left in range(sw - rw + 1):
                    lum_rect, c_rect = _lib.scaled_region_blocks(h, w, scale, top, left, rh, rw)
                    _check_cover(g, scale, top, left, rh, rw, lum_rect, c_rect)
                    shapes.add(lum_rect[2:] + c_rect[2:])
                    rows_l, rows_c = _taps(top, rh, nyc)
                    cols_l, cols_c = _taps(left, rw, nxc)
                    span = lambda s: int(s.max()) // m - int(s.min()) // m + 1
                    need = [max(a, b) for a, b in zip(need, (span(rows_l), span(cols_l), span(rows_c), span(cols_c)))]
            assert len(shapes) == 1, (rh, rw, shapes)
            (nyl, nxl, nyc_b, nxc_b), = shapes
            got = (nyl, nxl, nyc_b, nxc_b)
            assert all(a >= b for a, b in zip(got, need)) and all(a <= b + 1 for a, b in zip(got, need)), (got, need)
            for n in (1, 3):
                work, cap = _lib.scaled_region_sizes(n, h, w, scale, rh, rw)
                blocks = nyl * nxl + 2 * nyc_b * nxc_b
                assert cap == n * blocks
                assert work == -(-8 * n // 256) * 256 + n * m * m * blocks


def test_sizes_of_the_tiles():
    """112 x 112 of the 1/2 image and 56 x 56 of the 1/4 image of 640 x 426 (224 x 224 at full resolution); the 1/8
    window needs only its origins."""
    from hiccup_b200 import _lib
    g = _lib.geometry(426, 640)
    lum, c = _lib.scaled_region_blocks(426, 640, 2, 37, 101, 112, 112)
    assert lum[2:] == (29, 29) and c[2:] == (16, 16)
    lum, c = _lib.scaled_region_blocks(426, 640, 4, 0, 0, 56, 56)
    assert lum[2:] == (29, 29) and c[2:] == (16, 16)
    work, cap = _lib.scaled_region_sizes(1024, 426, 640, 2, 112, 112)
    assert cap == 1024 * (29 * 29 + 2 * 16 * 16) and work == 8192 + 16 * cap
    assert cap / (1024 * g.blocks_per_image) < 0.21
    work, cap = _lib.scaled_region_sizes(1024, 426, 640, 4, 56, 56)
    assert work == 8192 + 4 * cap
    assert _lib.scaled_region_sizes(1024, 426, 640, 8, 28, 28) == (8 * 1024, 0)


def test_library_refuses_bad_arguments():
    from hiccup_b200 import _lib
    lib = _lib.load()
    # 64 x 81: out 64 x 80; 1/2: 32 x 40, 1/4: 16 x 20, 1/8: 8 x 10
    for scale in (0, 1, 3, 8, 16, -2):
        with pytest.raises(_lib.HicError, match="error -1"):
            _lib.scaled_region_blocks(64, 81, scale, 0, 0, 1, 1)
    for scale in (0, 1, 3, 16):
        with pytest.raises(_lib.HicError, match="error -1"):
            _lib.scaled_region_sizes(1, 64, 81, scale, 1, 1)
    for scale, (sh, sw) in ((2, (32, 40)), (4, (16, 20)), (8, (8, 10))):
        bad = [(0, 0, 0, 1), (0, 0, 1, 0), (-1, 0, 1, 1), (0, -1, 1, 1), (sh, 0, 1, 1), (0, sw, 1, 1), (0, 0, sh + 1, 1),
               (0, 0, 1, sw + 1), (1, 0, sh, 1), (0, 1, 1, sw)]
        for top, left, rh, rw in bad:
            if scale != 8:
                with pytest.raises(_lib.HicError, match="error -1"):
                    _lib.scaled_region_blocks(64, 81, scale, top, left, rh, rw)
            if top == 0 and left == 0:
                with pytest.raises(_lib.HicError, match="error -1"):
                    _lib.scaled_region_sizes(2, 64, 81, scale, rh, rw)
        assert _lib.scaled_region_sizes(1, 64, 81, scale, sh, sw)[0] > 0
    with pytest.raises(_lib.HicError, match="error -1"):
        _lib.scaled_region_sizes(0, 64, 81, 2, 1, 1)
    # refused on the host before anything is launched: these pointers are never touched
    fake = 1 << 20
    for scale, (sh, sw) in ((2, (32, 40)), (4, (16, 20))):
        work, cap = _lib.scaled_region_sizes(2, 64, 81, scale, 4, 4)
        call = lambda coef=fake, sc=scale, o=np.zeros(4, np.int32), rh=4, rw=4, wk=fake, wb=work, ties=fake, stats=fake, out=fake: \
            lib.hic_dct_scaled_region(coef, 2, 64, 81, sc, None if o is None else o.ctypes.data, rh, rw, wk, wb, ties, cap,
                                      stats, out, None)
        for bad in (1, 3, 8):
            assert call(sc=bad) == -1 and b"scale" in lib.hic_last_error()
        for origin in ([0, 0, sh - 3, 0], [0, 0, 0, sw - 3], [-1, 0, 0, 0]):
            assert call(o=np.asarray(origin, np.int32)) == -1 and b"not inside" in lib.hic_last_error()
        assert call(rh=0) == -1 and b"empty" in lib.hic_last_error()
        assert call(wb=work - 1) == -1 and b"too small" in lib.hic_last_error()
        assert call(wk=fake + 8) == -1 and b"aligned" in lib.hic_last_error()
        assert call(coef=fake + 8) == -1 and b"aligned" in lib.hic_last_error()
        for kw in ({"coef": None}, {"o": None}, {"wk": None}, {"ties": None}, {"stats": None}, {"out": None}):
            assert call(**kw) == -1 and b"NULL" in lib.hic_last_error()
    work, cap = _lib.scaled_region_sizes(2, 64, 81, 8, 4, 4)
    assert (work, cap) == (16, 0)
    call = lambda dc=fake, o=np.zeros(4, np.int32), rh=4, rw=4, wk=fake, wb=work, out=fake: \
        lib.hic_dct_thumbnail_region(dc, 2, 64, 81, None if o is None else o.ctypes.data, rh, rw, wk, wb, out, None)
    for origin in ([0, 0, 5, 0], [0, 0, 0, 7], [0, -1, 0, 0]):
        assert call(o=np.asarray(origin, np.int32)) == -1 and b"not inside" in lib.hic_last_error()
    assert call(rw=0) == -1 and b"empty" in lib.hic_last_error()
    assert call(wb=work - 1) == -1 and b"too small" in lib.hic_last_error()
    assert call(wk=fake + 2) == -1 and b"aligned" in lib.hic_last_error()
    assert call(dc=fake + 1) == -1 and b"aligned" in lib.hic_last_error()
    for kw in ({"dc": None}, {"o": None}, {"wk": None}, {"out": None}):
        assert call(**kw) == -1 and b"NULL" in lib.hic_last_error()


def test_python_checks_scale_and_windows():
    from hiccup_b200 import _lib
    assert [_lib.region_scale_arg(s) for s in (1, 2, 4, np.int64(8))] == [1, 2, 4, 8]
    for bad in (0, 3, 16, 2.0, "2", True, None):
        with pytest.raises(ValueError):
            _lib.region_scale_arg(bad)
    # 64 x 81: out 64 x 80; 1/2: 32 x 40, 1/4: 16 x 20, 1/8: 8 x 10
    for scale, (sh, sw) in ((1, (64, 80)), (2, (32, 40)), (4, (16, 20)), (8, (8, 10))):
        good = _lib.region_origins(64, 81, [(0, 0), (sh - 2, sw - 2)], (2, 2), scale)
        assert good.dtype == np.int32 and good.shape == (2, 2)
        for origins, size in [([(sh - 1, 0)], (2, 2)), ([(0, sw - 1)], (2, 2)), ([(-1, 0)], (1, 1)), ([(0, 0)], (sh + 1, 1))]:
            with pytest.raises(ValueError, match="decoded image" if scale == 1 else "1/%d-scale" % scale):
                _lib.region_origins(64, 81, origins, size, scale)
        with pytest.raises(ValueError, match="empty"):
            _lib.region_origins(64, 81, [(0, 0)], (0, 1), scale)
    with pytest.raises(ValueError):
        _lib.region_origins(64, 81, [(0, 0)], (1, 1), 3)


def test_bad_scales_and_windows_are_refused_before_any_work(tmp_path):
    """jpeg_region with a bad scale or a window outside the 1/scale image raises ValueError, and with a wavelet file
    NotImplementedError, before a device is needed (this runs without one)."""
    from hiccup_b200 import codec, hicimage
    wp, dp = write_goldens(tmp_path)
    hi = hicimage.HicImage.from_file(dp)            # 64 x 64: 1/2 32 x 32, 1/4 16 x 16, 1/8 8 x 8
    for bad in (0, 3, 16, 2.0, "4", True):
        with pytest.raises(ValueError):
            codec.jpeg_region(hi, 0, 0, 1, 1, scale=bad)
    for scale, side in ((2, 32), (4, 16), (8, 8)):
        for top, left, rh, rw in [(0, 0, 0, 1), (0, 0, 1, 0), (-1, 0, 1, 1), (side, 0, 1, 1), (0, side - 1, 1, 2),
                                  (0, 0, side + 1, side)]:
            with pytest.raises(ValueError):
                codec.jpeg_region(hi, top, left, rh, rw, scale=scale)
        with pytest.raises(NotImplementedError, match="wavelet"):
            codec.jpeg_region(hicimage.HicImage.from_file(wp), 0, 0, 1, 1, scale=scale)
