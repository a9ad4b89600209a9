"""Region decode at reduced scale against the whole reduced decode, on one GPU (development aid; bench.py is the
contract).

    python tools/scaled_region_time.py [--reps 10] [--out profiles/r06_scaled_region_b200.json]

  C2 device-resident   DctBatchCodec(1024, 426, 640), from the encoder's own device output: decode_scaled_device(s)
                       against decode_regions_device(size, scale=s) with seeded windows of 112x112 (s = 2) and 56x56
                       (s = 4), and thumbnails_device() against 28x28 windows at s = 8 (CUDA events, after warm-up, the
                       two alternating); per-kernel times in a separate profiled pass, and the time per block of K7SR
                       against K7S
  C5 one file          16384^2: codec.jpeg_scaled / codec.jpeg_thumbnail against codec.jpeg_region(..., scale=s) of a
                       256x256 tile
Checks every window it times against the crop of the whole reduced decode.  Prints and writes one JSON line with the
card's name and power limit.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np

from region_time import kernels
from thumb_time import card, event_ms, host_ms

SIZES = {2: 112, 4: 56, 8: 28}          # C2: a 224 x 224 window of the full image, at each scale


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_scaled_region_b200.json"))
    args = ap.parse_args()
    import ctypes
    import torch
    import bench
    import bench_bands
    from hiccup_b200 import _lib, bands, codec
    from hiccup_b200.batch import DctBatchCodec
    _lib.require_device()
    buf = ctypes.create_string_buffer(256)
    _lib.check(_lib.load().hic_device_name(buf, len(buf)))
    res = {"tool": "scaled_region_time", "device": buf.value.decode(), "card": card(), "reps": args.reps}
    torch.cuda.init()
    checks = {}

    # ---- C2: 1024 x 640x426, the benchmark's images (seeds 2000..) ------------------------------------------------
    n, h, w = 1024, 426, 640
    base = bench.synthetic_batch(16, h, w, 2000)
    rgb = np.ascontiguousarray(base[np.arange(n) % 16])
    rgb[:, 0, :, 0] = (np.arange(n) // 16).astype(np.uint8)[:, None]            # 1024 distinct images
    bc = DctBatchCodec(n, h, w)
    bc.upload(rgb)
    enc = bc.encode_resident()
    res["c2_blocks"] = int(n * bc.g.blocks_per_image)
    for s, r in SIZES.items():
        sh, sw = bc.thumbnail_shape[1:3] if s == 8 else bc.scaled_shape(s)[1:3]
        rng = np.random.default_rng(1000 + s)
        origins = np.stack([rng.integers(0, sh - r + 1, n), rng.integers(0, sw - r + 1, n)], 1).astype(np.int32)
        whole_dev = bc.thumbnails_device if s == 8 else (lambda: bc.decode_scaled_device(s))
        region_dev = lambda: bc.decode_regions_device(origins, (r, r), scale=s)
        for _ in range(3):
            whole_dev()
            region_dev()
        torch.cuda.synchronize()
        whole, region = [], []
        for _ in range(3):                  # alternating windows
            whole.append(event_ms(whole_dev, args.reps))
            region.append(event_ms(region_dev, args.reps))
        key = "c2_s%d" % s
        res[key + "_whole_ms"] = statistics.median(whole)
        res[key + "_region_ms"] = statistics.median(region)
        res[key + "_windows_ms"] = {"whole": whole, "region": region}
        kw = res[key + "_whole_kernels_ms"] = kernels(whole_dev, args.reps)
        kr = res[key + "_region_kernels_ms"] = kernels(region_dev, args.reps)
        if s != 8:
            _, cap = _lib.scaled_region_sizes(n, h, w, s, r, r)
            res[key + "_region_blocks"] = int(cap)
            res[key + "_ns_per_block"] = {"scaled_inverse_kernel": 1e6 * kw["scaled_inverse_kernel"] / res["c2_blocks"],
                                          "scaled_region_inverse_kernel": 1e6 * kr["scaled_region_inverse_kernel"] / cap}
            names = ("scaled_inverse_kernel", "scaled_fixup_kernel", "scaled_colour_kernel")
            res[key + "_k7s_k8s_ms"] = round(sum(kw.get(k, 0.0) for k in names), 4)
            res[key + "_k7sr_k8sr_ms"] = round(sum(kr.get("scaled_region_" + k[len("scaled_"):], 0.0) for k in names), 4)
        want = (bc.thumbnails(enc) if s == 8 else bc.decode_scaled(enc, s)).copy()
        crops = np.stack([want[i, t:t + r, l:l + r] for i, (t, l) in enumerate(origins)])
        got = bc.decode_regions(enc, origins, (r, r), scale=s)
        region_dev()
        checks[key] = bool(np.array_equal(got, crops) and np.array_equal(bc.fetch_regions(), crops))
    bc.close()
    del rgb, base

    # ---- C5: one 16384^2 file, a 256 x 256 tile at an unaligned origin of each reduced image ----------------------
    size, tile = 16384, 256
    hic = bands.encode_banded(bench_bands.big_synthetic(size), 1)
    for s, (top, left) in ((2, (5003, 3777)), (4, (1501, 2999)), (8, (1001, 733))):
        whole_fn = (lambda: codec.jpeg_thumbnail(hic)) if s == 8 else (lambda: codec.jpeg_scaled(hic, s))
        region_fn = lambda: codec.jpeg_region(hic, top, left, tile, tile, scale=s)
        for _ in range(2):
            whole_fn()
            region_fn()
        whole, region = [], []
        for _ in range(3):
            whole.append(host_ms(whole_fn, 2))
            region.append(host_ms(region_fn, 2))
        key = "c5_s%d" % s
        res[key + "_whole_ms"] = statistics.median(whole)
        res[key + "_region_ms"] = statistics.median(region)
        res[key + "_windows_ms"] = {"whole": whole, "region": region}
        res[key + "_region_kernels_ms"] = kernels(region_fn, 2)
        checks[key] = bool(np.array_equal(region_fn(), whole_fn()[top:top + tile, left:left + tile]))
    res["checks_equal"] = checks
    res["card_after"] = card()

    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    if not all(checks.values()):
        sys.exit("a scaled region differs from the crop of the whole reduced decode: %r" % checks)


if __name__ == "__main__":
    main()
