"""Region decode against the full decode, on one GPU (development aid; bench.py is the contract).

    python tools/region_time.py [--reps 10] [--out profiles/r04_region_b200.json]

  C2 device-resident   DctBatchCodec(1024, 426, 640): decode_device() against decode_regions_device() with seeded
                       224x224 windows, from the encoder's own device output (CUDA events, after warm-up, the two
                       alternating); per-kernel times of both in a separate profiled pass, and the time per block
                       of K7R against K7
  C2 from .hic files   read_files() + decode() against read_files() + decode_regions() of the batch's 1024 files
                       (host clock: the calls end in a device synchronise)
  C5 one file          16384^2: codec.jpeg_decode + compression.jpeg_decompression against codec.jpeg_region of a
                       2048^2 window
Checks the batch windows against decode() cropped, and the C5 window against the full decode.  Prints and writes one
JSON line with the card's name and power limit.
"""
import argparse
import json
import os
import shutil
import statistics
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np

from thumb_time import card, event_ms, host_ms


def kernels(fn, reps):
    """Per-kernel mean ms per call of fn over reps profiled calls."""
    from hiccup_b200 import _lib
    _lib.profile_enable(True)
    _lib.profile_report()
    try:
        for _ in range(reps):
            fn()
        _lib.sync()
        rep = _lib.profile_report()
    finally:
        _lib.profile_enable(False)
    return {k: round(v[0] / reps, 4) for k, v in sorted(rep.items(), key=lambda kv: -kv[1][0])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_region_b200.json"))
    args = ap.parse_args()
    import ctypes
    import torch
    import bench
    import bench_bands
    from hiccup_b200 import _lib, bands, codec, compression
    from hiccup_b200.batch import DctBatchCodec
    _lib.require_device()
    buf = ctypes.create_string_buffer(256)
    _lib.check(_lib.load().hic_device_name(buf, len(buf)))
    res = {"tool": "region_time", "device": buf.value.decode(), "card": card(), "reps": args.reps}
    torch.cuda.init()

    # ---- C2: 1024 x 640x426, the benchmark's images (seeds 2000..), 224 x 224 windows ---------------------------
    n, h, w, rh, rw = 1024, 426, 640, 224, 224
    base = bench.synthetic_batch(16, h, w, 2000)
    rgb = np.ascontiguousarray(base[np.arange(n) % 16])
    rgb[:, 0, :, 0] = (np.arange(n) // 16).astype(np.uint8)[:, None]            # 1024 distinct images
    rng = np.random.default_rng(224)
    origins = np.stack([rng.integers(0, h - rh + 1, n), rng.integers(0, w - rw + 1, n)], 1).astype(np.int32)
    bc = DctBatchCodec(n, h, w)
    bc.upload(rgb)
    enc = bc.encode_resident()
    g = bc.g
    _, cap = _lib.region_sizes(n, h, w, rh, rw)
    res["c2_blocks"] = int(n * g.blocks_per_image)
    res["c2_region_blocks"] = int(cap)
    res["c2_region_pixel_share"] = rh * rw / (g.out_h * g.out_w)
    region_dev = lambda: bc.decode_regions_device(origins, (rh, rw))
    for _ in range(3):
        bc.decode_device()
        region_dev()
    torch.cuda.synchronize()
    full, region = [], []
    for _ in range(3):                      # alternating windows
        full.append(event_ms(bc.decode_device, args.reps))
        region.append(event_ms(region_dev, args.reps))
    res["c2_resident_decode_ms"] = statistics.median(full)
    res["c2_resident_region_ms"] = statistics.median(region)
    res["c2_resident_windows_ms"] = {"decode": full, "region": region}
    kr = res["c2_region_kernels_ms"] = kernels(region_dev, args.reps)
    kd = res["c2_decode_kernels_ms"] = kernels(bc.decode_device, args.reps)
    res["c2_ns_per_block"] = {"inverse_kernel": 1e6 * kd["inverse_kernel"] / res["c2_blocks"],
                              "region_inverse_kernel": 1e6 * kr["region_inverse_kernel"] / res["c2_region_blocks"]}
    want = bc.decode(enc).copy()
    got = bc.decode_regions(enc, origins, (rh, rw))
    res["c2_check_equal"] = all(np.array_equal(got[i], want[i, t:t + rh, l:l + rw]) for i, (t, l) in enumerate(origins))
    del want, got

    tmp = tempfile.mkdtemp(prefix="region_time_")
    try:
        paths = [os.path.join(tmp, "%04d.hic" % i) for i in range(n)]
        bc.write_files(enc, paths)
        out_full = np.empty(bc.out_shape, np.uint8)
        out_region = np.empty((n, rh, rw, 3), np.uint8)
        for _ in range(2):
            bc.decode(bc.read_files(paths), out=out_full)
            bc.decode_regions(bc.read_files(paths), origins, (rh, rw), out=out_region)
        full, region = [], []
        for _ in range(3):
            full.append(host_ms(lambda: bc.decode(bc.read_files(paths), out=out_full), max(2, args.reps // 3)))
            region.append(host_ms(lambda: bc.decode_regions(bc.read_files(paths), origins, (rh, rw), out=out_region),
                                  max(2, args.reps // 3)))
        res["c2_files_decode_ms"] = statistics.median(full)
        res["c2_files_region_ms"] = statistics.median(region)
        res["c2_files_windows_ms"] = {"decode": full, "region": region}
        res["c2_files_read_ms"] = host_ms(lambda: bc.read_files(paths), 3)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    bc.close()
    del rgb, base

    # ---- C5: one 16384^2 file, a 2048^2 window at an unaligned origin --------------------------------------------
    size, win, top, left = 16384, 2048, 5003, 7777
    hic = bands.encode_banded(bench_bands.big_synthetic(size), 1)
    for _ in range(2):
        compression.jpeg_decompression(codec.jpeg_decode(hic))
        codec.jpeg_region(hic, top, left, win, win)
    full, region = [], []
    for _ in range(3):
        full.append(host_ms(lambda: compression.jpeg_decompression(codec.jpeg_decode(hic)), 2))
        region.append(host_ms(lambda: codec.jpeg_region(hic, top, left, win, win), 2))
    res["c5_decode_ms"] = statistics.median(full)
    res["c5_region_ms"] = statistics.median(region)
    res["c5_windows_ms"] = {"decode": full, "region": region}
    res["c5_region_kernels_ms"] = kernels(lambda: codec.jpeg_region(hic, top, left, win, win), 2)
    res["c5_check_equal"] = bool(np.array_equal(codec.jpeg_region(hic, top, left, win, win),
                                                compression.jpeg_decompression(codec.jpeg_decode(hic))[top:top + win, left:left + win]))
    res["card_after"] = card()

    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    if not (res["c2_check_equal"] and res["c5_check_equal"]):
        sys.exit("region decode differs from the cropped full decode")


if __name__ == "__main__":
    main()
