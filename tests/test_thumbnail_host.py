"""Thumbnail decode, the parts that need no GPU: the closed form of a DC-only block, the thumbnail's shape, the
oracle thumbnail against an explicit block-by-block DC-only decode, the DC-stream gather of the batch path and
the command line."""
import os
import pickle

import numpy as np
import pytest

from oracle import hiccup_oracle as orc
from tests import thumbnail_oracle as tho
from tests.conftest import load_golden
from tests.reduced_helpers import DCT_GOLDENS


@pytest.mark.parametrize("table", ["lum", "chroma"])
def test_dc_only_block_closed_form_for_every_int16(table):
    """inv_dct_channel of a block whose only non-zero coefficient is its DC q is the constant
    ((q T00 + 32768) / 256 truncated toward zero) & 255 -- for every int16 q."""
    tab = orc.LUM_TABLE if table == "lum" else orc.CHROMA_TABLE
    t00 = int(np.asarray(tab)[0, 0])
    assert t00 == (16 if table == "lum" else 17)
    q = np.arange(-32768, 32768, dtype=np.int64)
    coefs = np.zeros((8, 8 * q.size), np.float64)
    coefs[0, ::8] = q
    pixels = orc.inv_dct_channel(coefs, tab).reshape(8, q.size, 8)
    assert (pixels == pixels[:1, :, :1]).all(), "a DC-only block is not constant"
    num = q * t00 + 32768
    closed = (np.sign(num) * (np.abs(num) // 256)) & 255            # C division: truncation toward zero
    assert np.array_equal(pixels[0, :, 0].astype(np.int64), closed)


SIZES = [(40, 40), (41, 41), (33, 47), (40, 41), (26, 40), (2, 2), (3, 5), (7, 9), (8, 8), (15, 17), (16, 16),
         (17, 33), (426, 640), (512, 512), (1080, 1920), (16384, 16384)] + [(h, w) for h in range(2, 70, 3) for w in (2, 31, 64)]


def test_thumbnail_shape_matches_the_library_and_the_bounds():
    from hiccup_b200 import _lib
    for h, w in SIZES:
        g = _lib.geometry(h, w)
        th, tw = _lib.thumbnail_shape(h, w)
        assert (th, tw) == tho.thumbnail_shape(h, w) == (-(-g.out_h // 8), -(-g.out_w // 8)), (h, w)
        assert th <= g.nby_l and th <= 2 * g.nby_c and tw <= g.nbx_l and tw <= 2 * g.nbx_c, (h, w)
    # the crop matters: h = 40 has five luminance block rows and six upsampled chroma rows, h = 41 six and six
    g40, g41 = _lib.geometry(40, 40), _lib.geometry(41, 41)
    assert (g40.nby_l, 2 * g40.nby_c, _lib.thumbnail_shape(40, 40)[0]) == (5, 6, 5)
    assert (g41.nby_l, 2 * g41.nby_c, _lib.thumbnail_shape(41, 41)[0]) == (6, 6, 5)
    with pytest.raises(_lib.HicError):
        _lib.thumbnail_shape(1, 8)


def _explicit_thumbnail(planes):
    """Block by block: each DC alone in an 8x8 coefficient block through inv_dct_channel, then pyr_up, crop, colour."""
    def values(plane, table):
        dc = tho.dc_terms(plane)
        out = np.zeros(dc.shape, np.uint8)
        for (by, bx), q in np.ndenumerate(dc):
            blk = np.zeros((8, 8))
            blk[0, 0] = q
            px = orc.inv_dct_channel(blk, table)
            assert (px == px[0, 0]).all()
            out[by, bx] = px[0, 0]
        return out
    h, w = np.asarray(planes["lum"]).shape
    th, tw = tho.thumbnail_shape(h, w)
    y = values(planes["lum"], orc.LUM_TABLE)[:th, :tw]
    cr = orc.pyr_up(values(planes["cr"], orc.CHROMA_TABLE))[:th, :tw]
    cb = orc.pyr_up(values(planes["cb"], orc.CHROMA_TABLE))[:th, :tw]
    return orc.ycrcb_to_rgb(y, cr, cb)


@pytest.mark.parametrize("name", DCT_GOLDENS)
def test_oracle_thumbnail_is_the_dc_only_decode(name):
    g = load_golden(name)
    planes = {ch: g["coef_" + ch] for ch in orc.CHANNELS}
    got = tho.jpeg_thumbnail(planes)
    h, w = planes["lum"].shape
    assert got.shape == tho.thumbnail_shape(h, w) + (3,) and got.dtype == np.uint8
    if name != "lenna512":                                  # 4096 + 2048 single-block transforms: the small ones suffice
        assert np.array_equal(got, _explicit_thumbnail(planes))
    # its luminance is the full DC-only decode's, sampled at the tiles' corners
    zero_ac = np.zeros_like(planes["lum"], np.float64)
    zero_ac[::8, ::8] = planes["lum"][::8, ::8]
    y_full = orc.inv_dct_channel(zero_ac, orc.LUM_TABLE)
    th, tw = got.shape[:2]
    assert np.array_equal(tho.dc_only_values(tho.dc_terms(planes["lum"]), orc.LUM_TABLE)[:th, :tw], y_full[::8, ::8][:th, :tw])


def test_dc_streams_only_gathers_the_dc_tables_and_bytes():
    from hiccup_b200 import entropy
    rng = np.random.default_rng(5)
    n_s = 9 * 2
    rows = rng.integers(0, 6, n_s).astype(np.uint32)
    start = np.concatenate(([0], np.cumsum(rows)[:-1])).astype(np.uint32)
    symbols = np.arange(int(rows.sum()), dtype=np.int32) * 7
    packed = rng.integers(0, 1 << 40, int(rows.sum()), dtype=np.uint64)
    byte_len = rng.integers(1, 11, n_s).astype(np.uint64)
    padded = (byte_len + np.uint64(3)) & ~np.uint64(3)
    byte_off = np.concatenate(([0], np.cumsum(padded)[:-1])).astype(np.uint64)
    data = rng.integers(0, 256, int(padded.sum()), dtype=np.uint8)
    nbits = rng.integers(1, 80, n_s).astype(np.uint64)
    enc = entropy.EncodedStreams(None, np.stack([start, rows], 1), None, nbits, byte_off, byte_len, symbols, packed, data)
    index, sym, pk, d, off, nb = entropy.dc_streams_only(enc)
    for s in range(n_s):
        if s % 3:
            assert index[s, 1] == 0 and nb[s] == 0
            continue
        a, n = int(index[s, 0]), int(index[s, 1])
        assert n == rows[s]
        assert np.array_equal(sym[a:a + n], symbols[start[s]:start[s] + n])
        assert np.array_equal(pk[a:a + n], packed[start[s]:start[s] + n])
        assert nb[s] == nbits[s] and int(off[s]) % 4 == 0
        o, L = int(off[s]), int(byte_len[s])
        assert d[o:o + L].tobytes() == enc.framed(s)
    assert sym.size == int(rows[0::3].sum()) and d.size == int(padded[0::3].sum()) + 16


def test_command_line(monkeypatch, tmp_path):
    from hiccup_b200 import run
    calls = []
    monkeypatch.setattr(run, "decompress", lambda path, save=None, thumbnail=False: calls.append(("one", path, save, thumbnail)))
    monkeypatch.setattr(run, "decompress_many", lambda paths, save_dir=None, max_batch=256, thumbnail=False:
                        calls.append(("many", list(paths), save_dir, thumbnail)))
    out = str(tmp_path)
    run.main(["-d", "x/a.hic", "-t", "-o", out])
    run.main(["--decompress", "a.hic", "b.hic", "--thumbnail", "-o", out])
    run.main(["-d", "a.hic", "-o", out])
    assert calls == [("one", "x/a.hic", os.path.join(out, "a.hic.thumb.png"), True),
                     ("many", ["a.hic", "b.hic"], out, True),
                     ("one", "a.hic", os.path.join(out, "a.hic.png"), False)]
    with pytest.raises(SystemExit):
        run.main(["-c", "img.png", "-t"])           # a thumbnail is a decode option


def test_wavelet_files_are_refused_before_any_work(tmp_path):
    """Wavelet files have no DC streams: every thumbnail entry point says so with NotImplementedError -- before it
    needs a device (this runs without one)."""
    from hiccup_b200 import codec, hicimage, run
    w = load_golden("w_syn64")
    d = load_golden("syn64")
    wp, dp = os.path.join(tmp_path, "w.hic"), os.path.join(tmp_path, "d.hic")
    with open(wp, "wb") as f:
        f.write(pickle.dumps(pickle.loads(w["hic"].tobytes())))
    with open(dp, "wb") as f:
        f.write(pickle.dumps(pickle.loads(d["hic"].tobytes())))
    with pytest.raises(NotImplementedError, match="wavelet"):
        codec.jpeg_thumbnail(hicimage.HicImage.from_file(wp))
    with pytest.raises(NotImplementedError, match="wavelet"):
        run.decompress(wp, thumbnail=True)
    with pytest.raises(NotImplementedError, match="wavelet"):
        run.decompress_many([dp, wp], save_dir=str(tmp_path), thumbnail=True)
    assert not [f for f in os.listdir(tmp_path) if f.endswith(".png")]
