"""Helpers the reduced-decode tests share (thumbnail, region, scaled, scaled region, wavelet scaled, restart records):
the kernels a call launches, the golden lists, golden files on disk, odd shapes, images that need the scaled fix-up
and the windows the region tests try."""
import os
import pickle

import numpy as np

from oracle import hiccup_oracle as orc
from tests.conftest import load_golden

# the DCT goldens of the reference, and those of them that also carry the reference's decoded pixels
DCT_GOLDENS = ["lenna512", "gh256", "syn64", "syn48x80", "syn64x106", "syn128x160", "syn26x40", "syn33x47",
               "tiny16", "flat32", "flat32b", "noise32x64"]
GOLDENS_WITH_PIXELS = ["flat32", "flat32b", "gh256", "lenna512", "noise32x64", "syn128x160", "syn48x80", "syn64", "tiny16"]

ODD = [(26, 40), (33, 47), (2, 2), (3, 5), (5, 3), (9, 17), (17, 2), (2, 31), (15, 15), (64, 106)]


def kernels_of(fn):
    """(fn(), the names of the kernels it launched)."""
    from hiccup_b200 import _lib
    _lib.profile_enable(True)
    _lib.profile_report()
    try:
        out = fn()
        _lib.sync()
        return out, set(_lib.profile_report())
    finally:
        _lib.profile_enable(False)


def planes(comp):
    """The three coefficient planes of a DCT-mode CompressedImage as arrays, by channel."""
    return {ch: np.asarray(v) for ch, v in comp.as_dict.items()}


def write_goldens(tmp_path):
    """The w_syn64 (wavelet) and syn64 (DCT) goldens as `.hic` files under tmp_path: (wavelet path, DCT path)."""
    wp, dp = os.path.join(tmp_path, "w.hic"), os.path.join(tmp_path, "d.hic")
    for path, name in ((wp, "w_syn64"), (dp, "syn64")):
        with open(path, "wb") as f:
            f.write(pickle.dumps(pickle.loads(load_golden(name)["hic"].tobytes())))
    return wp, dp


def tie_planes(h, w, scale, seed):
    """Large DC terms (samples that wrap) and large AC terms; the first blocks of every plane are ones whose float32
    samples truncate differently from the float64 definition -- found by K7S's arithmetic on the host (the CPU harness
    runs the same float32 code) -- so the fix-up must change samples."""
    from tests.test_scaled_host import _harness, _harness_blocks
    lib = _harness()
    rng = np.random.default_rng(seed)
    by_channel = {}
    for ch, shape in (("lum", (h, w)), ("cr", (h // 2, w // 2)), ("cb", (h // 2, w // 2))):
        nb = (shape[0] // 8) * (shape[1] // 8)
        pool = rng.integers(-1500, 1501, (200000, 64)) * (rng.random((200000, 64)) < 0.7)
        pool[:, 0] = rng.integers(-6000, 6000, len(pool))
        out, _, _, exact = _harness_blocks(lib, pool, 0 if ch == "lum" else 1, 8 // scale)
        miss = (out != exact).any(axis=1)
        zz = np.concatenate([pool[miss], pool[~miss]])[:nb]
        nat = np.zeros((nb, 64), np.int64)
        nat[:, orc.ZIGZAG8] = zz
        by_channel[ch] = orc.merge_blocks(nat.reshape(nb, 8, 8), shape).astype(np.int32)
    return by_channel


def fixed_windows(out_h, out_w):
    """Corners, edges, 1x1, single rows and columns, odd sizes at odd origins and the whole image."""
    wins = {(0, 0, out_h, out_w), (0, 0, 1, 1), (out_h - 1, out_w - 1, 1, 1), (0, out_w - 1, 1, 1), (out_h - 1, 0, 1, 1),
            (0, 0, 1, out_w), (out_h - 1, 0, 1, out_w), (0, 0, out_h, 1), (0, out_w - 1, out_h, 1)}
    for rh, rw in ((7, 9), (16, 16), (17, 33), (out_h // 2 + 1, out_w // 2 + 3), (out_h - 1, out_w - 1)):
        rh, rw = max(1, min(rh, out_h)), max(1, min(rw, out_w))
        for top in sorted({0, 1, (out_h - rh) // 2 | 1, out_h - rh}):
            for left in sorted({0, 3, (out_w - rw) // 2, out_w - rw}):
                if top + rh <= out_h and left + rw <= out_w:
                    wins.add((top, left, rh, rw))
    return sorted(wins)


def random_windows(out_h, out_w, rng):
    """Corners, edges, 1x1, single rows and columns, the whole image and a few random windows drawn from rng."""
    yield 0, 0, out_h, out_w
    for rh, rw in {(1, 1), (1, out_w), (out_h, 1), (min(7, out_h), min(9, out_w)), (min(16, out_h), min(16, out_w)),
                   (min(17, out_h), min(33, out_w)), ((out_h + 1) // 2, (out_w + 1) // 2)}:
        for top in {0, (out_h - rh) // 2, out_h - rh}:
            for left in {0, (out_w - rw) // 2, out_w - rw}:
                yield top, left, rh, rw
    for _ in range(12):
        rh, rw = int(rng.integers(1, out_h + 1)), int(rng.integers(1, out_w + 1))
        yield int(rng.integers(0, out_h - rh + 1)), int(rng.integers(0, out_w - rw + 1)), rh, rw
