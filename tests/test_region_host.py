"""Region decode, the parts that need no GPU: the block selection against a direct enumeration of what K8 reads, the
work and tie sizes, the argument checks of every entry point (they all refuse before any device work, so they run
here) and the command line."""
import os

import numpy as np
import pytest

from tests.reduced_helpers import random_windows, write_goldens

SIZES = [(2, 2), (3, 5), (5, 3), (2, 17), (17, 2), (3, 3), (7, 9), (8, 8), (9, 17), (15, 17), (16, 16), (17, 33),
         (26, 40), (33, 47), (40, 41), (64, 106), (96, 136), (426, 640)]


def _rows_read(top, rh, n_out, n_c):
    """Luminance rows and chroma rows K8 reads for output rows [top, top + rh) (the same rule for columns)."""
    lum, chroma = set(), set()
    for oy in range(top, top + rh):
        lum.add(oy)
        cy = oy >> 1
        ym = cy - 1 if cy > 0 else (1 if n_c > 1 else 0)
        yn = min(cy + 1, n_c - 1)
        chroma |= {ym, cy, yn}
    return lum, chroma


def _check_cover(g, top, left, rh, rw, lum_rect, c_rect):
    rows_l, rows_c = _rows_read(top, rh, g.out_h, g.hc)
    cols_l, cols_c = _rows_read(left, rw, g.out_w, g.wc)
    by, bx, nby, nbx = lum_rect
    assert 0 <= by and by + nby <= g.nby_l and 0 <= bx and bx + nbx <= g.nbx_l
    assert all(by <= r // 8 < by + nby for r in rows_l) and all(bx <= c // 8 < bx + nbx for c in cols_l)
    assert all(r < g.h for r in rows_l) and all(c < g.w for c in cols_l)
    by, bx, nby, nbx = c_rect
    assert 0 <= by and by + nby <= g.nby_c and 0 <= bx and bx + nbx <= g.nbx_c
    assert all(0 <= r < g.hc and by <= r // 8 < by + nby for r in rows_c)
    assert all(0 <= c < g.wc and bx <= c // 8 < bx + nbx for c in cols_c)


@pytest.mark.parametrize("h,w", SIZES)
def test_selection_covers_every_sample_k8_reads(h, w):
    from hiccup_b200 import _lib
    g = _lib.geometry(h, w)
    rng = np.random.default_rng(h * 1000 + w)
    for top, left, rh, rw in random_windows(g.out_h, g.out_w, rng):
        lum_rect, c_rect = _lib.region_blocks(h, w, top, left, rh, rw)
        _check_cover(g, top, left, rh, rw, lum_rect, c_rect)


@pytest.mark.parametrize("h,w", [(2, 2), (3, 5), (5, 3), (9, 17), (17, 33), (26, 40), (33, 47)])
def test_every_origin_of_every_size(h, w):
    """Every window of every size of a small image (a spread of sizes in the larger ones): covered, and every
    origin of one size selects rectangles of one size -- the most blocks any origin needs -- which is what
    hic_dct_region_sizes counts."""
    from hiccup_b200 import _lib
    g = _lib.geometry(h, w)
    pick = lambda n: range(1, n + 1) if n <= 16 else sorted({1, 2, 3, 7, 8, 9, 15, 16, 17, 18, n - 1, n})
    for rh in pick(g.out_h):
        for rw in pick(g.out_w):
            shapes, need = set(), [0, 0, 0, 0]
            for top in range(g.out_h - rh + 1):
                for left in range(g.out_w - rw + 1):
                    lum_rect, c_rect = _lib.region_blocks(h, w, top, left, rh, rw)
                    _check_cover(g, top, left, rh, rw, lum_rect, c_rect)
                    shapes.add(lum_rect[2:] + c_rect[2:])
                    rows_l, rows_c = _rows_read(top, rh, g.out_h, g.hc)
                    cols_l, cols_c = _rows_read(left, rw, g.out_w, g.wc)
                    span = lambda s: max(s) // 8 - min(s) // 8 + 1
                    need = [max(a, b) for a, b in zip(need, (span(rows_l), span(cols_l), span(rows_c), span(cols_c)))]
            assert len(shapes) == 1, (rh, rw, shapes)
            (nyl, nxl, nyc, nxc), = shapes
            # never fewer blocks than the worst origin needs, and at most one more per axis
            assert nyl >= need[0] and nxl >= need[1] and nyc >= need[2] and nxc >= need[3]
            assert nyl <= need[0] + 1 and nxl <= need[1] + 1 and nyc <= need[2] + 1 and nxc <= need[3] + 1
            for n in (1, 3):
                work, cap = _lib.region_sizes(n, h, w, rh, rw)
                blocks = nyl * nxl + 2 * nyc * nxc
                assert cap == n * blocks
                assert work >= 8 * n + 64 * n * blocks


def test_sizes_of_the_c2_crop():
    """224 x 224 out of 640 x 426: at most 29 x 29 luminance blocks and 16 x 16 per chroma plane."""
    from hiccup_b200 import _lib
    lum, c = _lib.region_blocks(426, 640, 37, 101, 224, 224)
    assert lum[2:] == (29, 29) and c[2:] == (16, 16)
    work, cap = _lib.region_sizes(1024, 426, 640, 224, 224)
    assert cap == 1024 * (29 * 29 + 2 * 16 * 16)
    assert work == 1024 * 64 * cap // 1024 + 8192
    g = _lib.geometry(426, 640)
    assert cap / (1024 * g.blocks_per_image) < 0.21


def test_library_refuses_bad_windows():
    from hiccup_b200 import _lib
    lib = _lib.load()
    for top, left, rh, rw in [(0, 0, 0, 5), (0, 0, 5, 0), (-1, 0, 4, 4), (0, -1, 4, 4), (61, 0, 4, 4), (0, 77, 4, 4),
                              (0, 0, 65, 4), (0, 0, 4, 81)]:
        with pytest.raises(_lib.HicError, match="error -1"):
            _lib.region_blocks(64, 81, top, left, rh, rw)          # out_h x out_w = 64 x 80
    with pytest.raises(_lib.HicError, match="error -1"):
        _lib.region_sizes(2, 64, 81, 65, 4)
    with pytest.raises(_lib.HicError, match="error -1"):
        _lib.region_sizes(2, 64, 81, 4, 0)
    work, cap = _lib.region_sizes(2, 64, 81, 8, 8)
    # the origins are checked on the host before anything is launched: these pointers are never touched
    fake = 1 << 20
    for origin in ([0, 0, 57, 0], [0, 0, 0, 73], [-1, 0, 0, 0]):
        o = np.asarray(origin, np.int32)
        rc = lib.hic_dct_region(fake, 2, 64, 81, o.ctypes.data, 8, 8, fake, work, fake, cap, fake, fake, None)
        assert rc == -1 and b"not inside" in lib.hic_last_error()
    o = np.zeros(4, np.int32)
    assert lib.hic_dct_region(fake, 2, 64, 81, o.ctypes.data, 8, 8, fake, work - 1, fake, cap, fake, fake, None) == -1
    assert lib.hic_dct_region(fake, 2, 64, 81, None, 8, 8, fake, work, fake, cap, fake, fake, None) == -1


def test_python_checks_windows():
    from hiccup_b200 import _lib
    good = _lib.region_origins(64, 81, [(0, 0), (56, 72)], (8, 8))
    assert good.dtype == np.int32 and good.shape == (2, 2) and good.flags.c_contiguous
    for origins, size in [([(0, 0), (57, 0)], (8, 8)), ([(0, 73)], (8, 8)), ([(-1, 0)], (8, 8)), ([(0, 0)], (0, 8)),
                          ([(0, 0)], (8, 0)), ([(0, 0)], (65, 1)), (np.zeros((0, 2), np.int32), (1, 1)),
                          ([0, 0], (1, 1)), ([(0.0, 0.0)], (1, 1))]:
        with pytest.raises(ValueError):
            _lib.region_origins(64, 81, origins, size)


def test_bad_windows_are_refused_before_any_work(tmp_path):
    """An empty window or one the 64 x 64 image does not hold: ValueError from every entry point, before a device is
    needed (this runs without one) and before any file is written."""
    from hiccup_b200 import codec, hicimage, run
    _, dp = write_goldens(tmp_path)
    hi = hicimage.HicImage.from_file(dp)
    for top, left, rh, rw in [(0, 0, 0, 4), (0, 0, 4, 0), (-1, 0, 4, 4), (0, -2, 4, 4), (61, 0, 4, 4), (0, 0, 65, 64),
                              (0, 60, 1, 5)]:
        with pytest.raises(ValueError):
            codec.jpeg_region(hi, top, left, rh, rw)
        with pytest.raises(ValueError):
            run.decompress(dp, save=os.path.join(tmp_path, "x.png"), region=(top, left, rh, rw))
        with pytest.raises(ValueError):
            run.decompress_many([dp, dp], save_dir=str(tmp_path), region=(top, left, rh, rw))
    for bad in [(0, 0, 4), (0, 0, 4, 4, 4), (0, 0, 4.0, 4)]:
        with pytest.raises(ValueError):
            run.decompress(dp, region=bad)
    with pytest.raises(ValueError, match="thumbnail"):
        run.decompress(dp, thumbnail=True, region=(0, 0, 4, 4))
    with pytest.raises(ValueError, match="thumbnail"):
        run.decompress_many([dp], save_dir=str(tmp_path), thumbnail=True, region=(0, 0, 4, 4))
    assert not [f for f in os.listdir(tmp_path) if f.endswith(".png")]


def test_wavelet_files_are_refused_before_any_work(tmp_path):
    from hiccup_b200 import codec, hicimage, run
    wp, dp = write_goldens(tmp_path)
    with pytest.raises(NotImplementedError, match="wavelet"):
        codec.jpeg_region(hicimage.HicImage.from_file(wp), 0, 0, 4, 4)
    with pytest.raises(NotImplementedError, match="wavelet"):
        run.decompress(wp, save=os.path.join(tmp_path, "w.png"), region=(0, 0, 4, 4))
    with pytest.raises(NotImplementedError, match="wavelet"):
        run.decompress_many([dp, wp], save_dir=str(tmp_path), region=(0, 0, 4, 4))
    assert not [f for f in os.listdir(tmp_path) if f.endswith(".png")]


def test_command_line(monkeypatch, tmp_path, capsys):
    from hiccup_b200 import run
    calls = []
    monkeypatch.setattr(run, "decompress", lambda path, save=None, thumbnail=False, region=None:
                        calls.append(("one", path, save, thumbnail, region)))
    monkeypatch.setattr(run, "decompress_many", lambda paths, save_dir=None, max_batch=256, thumbnail=False, region=None:
                        calls.append(("many", list(paths), save_dir, thumbnail, region)))
    out = str(tmp_path)
    run.main(["-d", "x/a.hic", "--region", "1,2,30,40", "-o", out])
    run.main(["--decompress", "a.hic", "b.hic", "--region", "0,0,8,8", "-o", out])
    run.main(["-d", "a.hic", "-o", out])
    assert calls == [("one", "x/a.hic", os.path.join(out, "a.hic.region.png"), False, (1, 2, 30, 40)),
                     ("many", ["a.hic", "b.hic"], out, False, (0, 0, 8, 8)),
                     ("one", "a.hic", os.path.join(out, "a.hic.png"), False, None)]
    printed = capsys.readouterr().out.split()
    assert printed[:3] == [os.path.join(out, "a.hic.region.png"), os.path.join(out, "a.hic.region.png"),
                           os.path.join(out, "b.hic.region.png")]
    for argv in (["-c", "img.png", "--region", "0,0,8,8"],             # a region is a decode option
                 ["-d", "a.hic", "-t", "--region", "0,0,8,8"],          # and not a thumbnail one
                 ["-d", "a.hic", "--region", "0,0,8"],
                 ["-d", "a.hic", "--region", "0,0,8,x"]):
        with pytest.raises(SystemExit):
            run.main(argv)
    assert len(calls) == 3
