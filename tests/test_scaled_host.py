"""Scaled decode, the parts that need no GPU: the committed basis against its closed form and the tile-mean property,
the oracle at m = 1 against the thumbnail, the float64 arithmetic the fix-up kernel runs (CPU harness) against the
oracle, the float32 path's flagging and error bound, the shapes, the argument checks of every entry point and the
command line."""
import ctypes
import os

import numpy as np
import pytest

from oracle import hiccup_oracle as orc
from tests import scaled_oracle as so
from tests import thumbnail_oracle as tho
from tests.conftest import load_golden
from tests.reduced_helpers import DCT_GOLDENS, write_goldens
from tests.test_oracle_dct import _ptr

HARNESS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "cpu_harness", "libhic_scaled_harness.so")


def _harness():
    if not os.path.exists(HARNESS):
        import __graft_entry__
        __graft_entry__.build()
    return ctypes.CDLL(HARNESS)

TABLES = {0: orc.LUM_TABLE, 1: orc.CHROMA_TABLE}


@pytest.mark.parametrize("scale", [2, 4])
def test_basis_is_the_closed_form(scale):
    m = 8 // scale
    b = so.BASIS[m]
    assert (b[:, 0] == 1.0).all()
    assert np.array_equal(b, so.closed_form_basis(scale))               # correctly rounded: within half an ulp
    lib = _harness()
    committed = np.zeros(m * m)
    lib.hx_scaled_basis(m, _ptr(committed))
    assert np.array_equal(committed.reshape(m, m), b)                  # csrc/hic_core.cuh holds the same bits
    if scale == 2:
        assert np.allclose(b[0], [1, 1.81225489, 1.30656296, 0.63637929], atol=1e-8)
    else:
        assert np.allclose(b, [[1, 1.28145772], [1, -1.28145772]], atol=1e-8)


@pytest.mark.parametrize("scale", [2, 4])
def test_tile_means_of_the_full_idct(scale):
    """B X B^T is the mean of each s x s tile of the unrounded 8 x 8 IDCT of a block with coefficients only at u, v < m."""
    m = 8 // scale
    rng = np.random.default_rng(scale)
    x = np.zeros((2000, 8, 8))
    x[:, :m, :m] = rng.integers(-3000, 3001, (2000, m, m))
    full = np.swapaxes(orc.ducc_dct3_8(np.swapaxes(orc.ducc_dct3_8(x), -1, -2)), -1, -2)
    means = full.reshape(-1, m, scale, m, scale).mean(axis=(2, 4))
    b = so.BASIS[m]
    reduced = b @ x[:, :m, :m] @ b.T
    assert np.abs(reduced - means).max() <= 1e-9 * max(1.0, np.abs(means).max())


@pytest.mark.parametrize("name", DCT_GOLDENS)
def test_m1_is_the_thumbnail(name):
    g = load_golden(name)
    planes = {ch: g["coef_" + ch] for ch in orc.CHANNELS}
    h, w = planes["lum"].shape
    m1 = orc.ycrcb_to_rgb(*(p[:tho.thumbnail_shape(h, w)[0], :tho.thumbnail_shape(h, w)[1]] for p in (
        so.scaled_plane(planes["lum"], orc.LUM_TABLE, 1), orc.pyr_up(so.scaled_plane(planes["cr"], orc.CHROMA_TABLE, 1)),
        orc.pyr_up(so.scaled_plane(planes["cb"], orc.CHROMA_TABLE, 1)))))
    assert np.array_equal(m1, tho.jpeg_thumbnail(planes))
    for scale in (2, 4):
        got = so.jpeg_scaled(planes, scale)
        assert got.shape == so.scaled_shape(h, w, scale) + (3,) and got.dtype == np.uint8


def _harness_blocks(lib, zz, kind, m):
    zz = np.ascontiguousarray(zz.reshape(-1, 64).astype(np.int16))
    nb = len(zz)
    out, exact = np.zeros((nb, m * m), np.uint8), np.zeros((nb, m * m), np.uint8)
    flagged, ratio = np.zeros(nb, np.uint8), np.zeros(nb)
    lib.hx_scaled_blocks(_ptr(zz), nb, kind, m, _ptr(out), _ptr(flagged), _ptr(ratio), _ptr(exact))
    return out, flagged.astype(bool), ratio, exact


def _oracle_blocks(zz, kind, m):
    nat = np.zeros((len(zz), 64), np.int64)
    nat[:, orc.ZIGZAG8] = zz
    return orc.astype_u8(so.block_values(nat.reshape(-1, 8, 8), TABLES[kind], m)).reshape(len(zz), m * m)


@pytest.mark.parametrize("scale", [2, 4])
@pytest.mark.parametrize("kind", [0, 1])
def test_float64_definition_matches_the_oracle(scale, kind):
    """The fix-up kernel's float64 arithmetic (scaled_decoded_block, through the CPU harness) equals the oracle bit for
    bit on a million random blocks per scale and table: small and large values, sparse blocks and int16 extremes."""
    m = 8 // scale
    lib = _harness()
    rng = np.random.default_rng(100 * scale + kind)
    n = 250000
    pools = [rng.integers(-40, 41, (n, 64)),
             rng.integers(-32768, 32768, (n, 64)),
             rng.integers(-2000, 2001, (n, 64)) * (rng.random((n, 64)) < 0.3),
             rng.choice([-32768, 32767, -1, 0, 1], (n, 64))]
    for pool in pools:
        zz = pool.astype(np.int16)
        _, _, _, exact = _harness_blocks(lib, zz, kind, m)
        assert np.array_equal(exact, _oracle_blocks(zz.astype(np.int64), kind, m))


@pytest.mark.parametrize("scale", [2, 4])
@pytest.mark.parametrize("kind", [0, 1])
def test_float32_near_integers_are_all_flagged(scale, kind, capsys):
    """K7S's float32 path on the host: every block whose truncated samples differ from the float64 definition is
    flagged, over random blocks and blocks from real images, then hill climbing towards the bound; the worst observed
    error stays below the rigorous bound (ratio < 1)."""
    m = 8 // scale
    lib = _harness()
    rng = np.random.default_rng(7 * scale + kind)
    n = 100000

    def run(zz):
        out, flagged, ratio, exact = _harness_blocks(lib, zz, kind, m)
        miss = (out != exact).any(axis=1)
        assert not (miss & ~flagged).any()
        return ratio, miss

    ch = "lum" if kind == 0 else "cr"
    real = np.concatenate([orc.blocks_zigzag(orc.jpeg_compression(orc.synthetic_image(128, 192, s))[ch]) for s in (11, 12)])
    pools = [real,
             rng.integers(-30, 31, (n, 64)),
             rng.integers(-600, 601, (n, 64)) * (rng.random((n, 64)) < 0.3),
             rng.integers(-3, 4, (n, 64)) + 900 * (np.arange(64)[None, :] == rng.integers(0, 2 * m * m, (n, 1))),
             rng.integers(-32768, 32768, (n, 64))]
    best, misses = 0.0, 0
    for pool in pools:
        pool = np.clip(pool, -32768, 32767)
        ratio, miss = run(pool)
        misses += int(miss.sum())
        best = max(best, float(ratio.max()))
        cur = pool[np.argsort(ratio)[-64:]].copy()
        cur_r = np.sort(ratio)[-64:].copy()
        for _ in range(60):
            cand = cur.copy()
            idx = rng.integers(0, 25 if m == 4 else 5, (64, 2))
            cand[np.arange(64)[:, None], idx] = np.clip(cand[np.arange(64)[:, None], idx] + rng.integers(-40, 41, (64, 2)),
                                                       -32768, 32767)
            r, _ = run(cand)
            better = r > cur_r
            cur[better], cur_r[better] = cand[better], r[better]
        best = max(best, float(cur_r.max()))
    with capsys.disabled():
        print("\n[scaled s=%d kind=%d] worst observed float32 error / rigorous bound: %.3f (%d float32 misses, all flagged)"
              % (scale, kind, best, misses))
    assert best < 1.0


SIZES = [(h, w) for h in range(2, 301, 7) for w in (2, 3, 17, 64, 299, 300)] + [(300, 300), (16384, 16384), (426, 640)]


def test_shapes_fit_the_reduced_planes():
    from hiccup_b200 import _lib
    for h, w in SIZES:
        g = _lib.geometry(h, w)
        for scale in (2, 4):
            m = 8 // scale
            sh, sw = _lib.scaled_shape(h, w, scale)
            assert (sh, sw) == so.scaled_shape(h, w, scale) == (-(-g.out_h // scale), -(-g.out_w // scale)), (h, w, scale)
            assert sh <= m * g.nby_l and sh <= 2 * m * g.nby_c and sw <= m * g.nbx_l and sw <= 2 * m * g.nbx_c, (h, w)
            work, cap = _lib.scaled_sizes(3, h, w, scale)
            assert cap == 3 * g.blocks_per_image and work == 3 * g.blocks_per_image * m * m
    assert _lib.scaled_shape(426, 640, 2) == (213, 320) and _lib.scaled_shape(426, 640, 4) == (107, 160)


def test_library_refuses_bad_arguments():
    from hiccup_b200 import _lib
    lib = _lib.load()
    for scale in (0, 1, 3, 8, 16, -2):
        with pytest.raises(_lib.HicError, match="error -1"):
            _lib.scaled_shape(64, 64, scale)
        with pytest.raises(_lib.HicError, match="error -1"):
            _lib.scaled_sizes(1, 64, 64, scale)
    with pytest.raises(_lib.HicError, match="error -1"):
        _lib.scaled_shape(1, 8, 2)
    with pytest.raises(_lib.HicError, match="error -1"):
        _lib.scaled_sizes(0, 64, 64, 2)
    work, cap = _lib.scaled_sizes(2, 64, 81, 2)
    # refused on the host before anything is launched: these pointers are never touched
    fake = 1 << 20
    for scale in (1, 3, 8):
        assert lib.hic_dct_scaled(fake, 2, 64, 81, scale, fake, work, fake, cap, fake, fake, None) == -1
        assert b"scale" in lib.hic_last_error()
    assert lib.hic_dct_scaled(fake, 2, 64, 81, 2, fake, work - 1, fake, cap, fake, fake, None) == -1
    assert lib.hic_dct_scaled(fake, 2, 64, 81, 2, fake + 8, work, fake, cap, fake, fake, None) == -1
    assert lib.hic_dct_scaled(None, 2, 64, 81, 2, fake, work, fake, cap, fake, fake, None) == -1


def test_python_checks_the_scale():
    from hiccup_b200 import _lib
    assert _lib.scale_arg(2) == 2 and _lib.scale_arg(np.int64(4)) == 4
    for bad in (1, 3, 8, 2.0, "2", True, None):
        with pytest.raises(ValueError):
            _lib.scale_arg(bad)


def test_bad_scales_and_wavelet_files_are_refused_before_any_work(tmp_path):
    """A scale other than 2 or 4 raises ValueError and a wavelet file NotImplementedError from every entry point, before
    a device is needed (this runs without one) and before any file is written."""
    from hiccup_b200 import codec, hicimage, run
    wp, dp = write_goldens(tmp_path)
    hi = hicimage.HicImage.from_file(dp)
    for bad in (1, 3, 8, 2.5):
        with pytest.raises(ValueError):
            codec.jpeg_scaled(hi, bad)
        with pytest.raises(ValueError):
            run.decompress(dp, save=os.path.join(tmp_path, "x.png"), scale=bad)
        with pytest.raises(ValueError):
            run.decompress_many([dp, dp], save_dir=str(tmp_path), scale=bad)
    with pytest.raises(ValueError, match="thumbnail"):
        run.decompress(dp, thumbnail=True, scale=2)
    with pytest.raises(ValueError, match="region"):
        run.decompress_many([dp], save_dir=str(tmp_path), region=(0, 0, 4, 4), scale=4)
    with pytest.raises(NotImplementedError, match="wavelet"):
        codec.jpeg_scaled(hicimage.HicImage.from_file(wp), 2)
    with pytest.raises(NotImplementedError, match="wavelet"):
        run.decompress(wp, save=os.path.join(tmp_path, "w.png"), scale=2)
    with pytest.raises(NotImplementedError, match="wavelet"):
        run.decompress_many([dp, wp], save_dir=str(tmp_path), scale=4)
    assert not [f for f in os.listdir(tmp_path) if f.endswith(".png")]


def test_command_line(monkeypatch, tmp_path, capsys):
    from hiccup_b200 import run
    calls = []
    monkeypatch.setattr(run, "decompress", lambda path, save=None, thumbnail=False, region=None, scale=None:
                        calls.append(("one", path, save, thumbnail, region, scale)))
    monkeypatch.setattr(run, "decompress_many", lambda paths, save_dir=None, max_batch=256, thumbnail=False, region=None,
                        scale=None: calls.append(("many", list(paths), save_dir, thumbnail, region, scale)))
    out = str(tmp_path)
    run.main(["-d", "x/a.hic", "--scale", "2", "-o", out])
    run.main(["--decompress", "a.hic", "b.hic", "--scale", "4", "-o", out])
    run.main(["-d", "a.hic", "-o", out])
    assert calls == [("one", "x/a.hic", os.path.join(out, "a.hic.s2.png"), False, None, 2),
                     ("many", ["a.hic", "b.hic"], out, False, None, 4),
                     ("one", "a.hic", os.path.join(out, "a.hic.png"), False, None, None)]
    printed = capsys.readouterr().out.split()
    assert printed[:3] == [os.path.join(out, "a.hic.s2.png"), os.path.join(out, "a.hic.s4.png"),
                           os.path.join(out, "b.hic.s4.png")]
    for argv in (["-c", "img.png", "--scale", "2"],                   # a scale is a decode option
                 ["-d", "a.hic", "-t", "--scale", "2"],                # and goes neither with a thumbnail
                 ["-d", "a.hic", "--region", "0,0,8,8", "--scale", "4"],   # nor with a region
                 ["-d", "a.hic", "--scale", "8"],
                 ["-d", "a.hic", "--scale", "3"],
                 ["-d", "a.hic", "--scale", "x"]):
        with pytest.raises(SystemExit):
            run.main(argv)
    assert len(calls) == 3
