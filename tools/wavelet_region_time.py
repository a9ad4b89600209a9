"""Wavelet region decode (hic_wavelet_region) against the full and scaled decodes it replaces, on one GPU (development
aid; bench.py is the contract).

    python tools/wavelet_region_time.py [--reps 10] [--out profiles/r08_wavelet_region_b200.json]

  C4 device-resident     WaveletBatchCodec(1, 4320, 7680), the benchmark's image: decode_device() against
                         decode_regions_device() of a 1920x1080 window at scale 1 and of a 256x256 tile at scales 1, 2, 4
                         and 8, from the encoder's own device output (CUDA events, after warm-up; each window is timed in
                         alternation with decode_device, medians of three windows); per-kernel times in a profiled pass
  C4 from its .hic file  codec.wavelet_region against codec.wavelet_decode + compression.wavelet_decompression + crop and
                         against codec.wavelet_scaled + crop (host clock: the calls end in a device synchronise)
  batch device-resident  WaveletBatchCodec(1024, 432, 640): seeded 224x224 windows per image at scale 1 and the same
                         windows at scales 2, 4 and 8 (origin and size divided by the scale)
Every timed window is checked against the crop it replaces.  Prints and writes one JSON line with the card's name, power
limit and max SM clock, read before and after.
"""
import argparse
import ctypes
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np

from region_time import kernels
from thumb_time import card, host_ms
from wavelet_scaled_time import alternate


def crops(img, origins, rh, rw):
    return np.stack([img[i, t:t + rh, l:l + rw] for i, (t, l) in enumerate(np.asarray(origins).tolist())])


def resident(bc, windows, reps, res, tag):
    """decode_device against decode_regions_device for each (name, origins, (rh, rw), scale); windows checked against
    crops of fetch() (scale 1) or fetch_scaled()."""
    bc.decode_device()
    ref = {1: bc.fetch().copy()}
    times, wins, kern, checks = {}, {}, {}, {}
    kern["decode"] = kernels(bc.decode_device, reps)
    for name, origins, size, s in windows:
        if s not in ref:
            bc.decode_scaled_device(s)
            ref[s] = bc.fetch_scaled().copy()
        region = lambda: bc.decode_regions_device(origins, size, scale=s)
        med, win = alternate({"decode": bc.decode_device, name: region}, reps)
        times[name], wins[name] = {"decode": med["decode"], "region": med[name]}, win
        kern[name] = kernels(region, reps)
        region()
        checks[name] = bool(np.array_equal(bc.fetch_regions(), crops(ref[s], origins, *size)))
    res[tag + "_resident_ms"], res[tag + "_resident_windows_ms"] = times, wins
    res[tag + "_kernels_ms"] = kern
    res[tag + "_check_windows_equal_crops"] = all(checks.values())
    res[tag + "_checks"] = checks


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_wavelet_region_b200.json"))
    args = ap.parse_args()
    import torch
    import bench
    from hiccup_b200 import _lib, codec, compression
    from hiccup_b200.batch import WaveletBatchCodec
    _lib.require_device()
    buf = ctypes.create_string_buffer(256)
    _lib.check(_lib.load().hic_device_name(buf, len(buf)))
    res = {"tool": "wavelet_region_time", "device": buf.value.decode(), "card": card(), "reps": args.reps}
    torch.cuda.init()

    # ---- C4: one 7680x4320 image, the benchmark's (seed 2000) -------------------------------------------------------
    h, w = 4320, 7680
    rgb = bench.synthetic_batch(1, h, w, 2000)
    bc = WaveletBatchCodec(1, h, w)
    bc.upload(rgb)
    enc = bc.encode_resident()
    hic = bc.hic_images(enc)[0]
    windows = [("w1920x1080_s1", [(1601, 2883)], (1080, 1920), 1)]
    windows += [("t256_s%d" % s, [(1601 // s, 2883 // s)], (256, 256), s) for s in (1, 2, 4, 8)]
    res["c4_windows"] = {name: {"origin": o[0], "size": list(size), "scale": s} for name, o, size, s in windows}
    resident(bc, windows, args.reps, res, "c4")

    def crop(img, o, size):
        return img[o[0]:o[0] + size[0], o[1]:o[1] + size[1]]

    calls, checks = {}, {}
    for name, (o,), size, s in windows:
        calls[name] = (lambda o=o, size=size, s=s: codec.wavelet_region(hic, o[0], o[1], size[0], size[1], s))
        if s == 1:
            calls[name + "_via_decode"] = (lambda o=o, size=size: crop(compression.wavelet_decompression(codec.wavelet_decode(hic)), o, size).copy())
        else:
            calls[name + "_via_scaled"] = (lambda o=o, size=size, s=s: crop(codec.wavelet_scaled(hic, s), o, size).copy())
    for fn in calls.values():
        fn()
    wins = {k: [] for k in calls}
    for _ in range(3):
        for k, fn in calls.items():
            wins[k].append(host_ms(fn, max(2, args.reps // 3)))
    res["c4_file_ms"] = {k: statistics.median(v) for k, v in wins.items()}
    res["c4_file_windows_ms"] = wins
    res["c4_file_kernels_ms"] = {k: kernels(fn, 2) for k, fn in calls.items()}
    for name, (o,), size, s in windows:
        checks[name] = bool(np.array_equal(calls[name](), calls[name + ("_via_decode" if s == 1 else "_via_scaled")]()))
    res["c4_check_file_windows_equal_crops"] = all(checks.values())
    bc.close()
    del rgb

    # ---- a batch: 1024 x 432x640, seeded 224x224 windows ---------------------------------------------------------------
    n, h, w = 1024, 432, 640
    base = bench.synthetic_batch(16, h, w, 2000)
    rgb = np.ascontiguousarray(base[np.arange(n) % 16])
    rgb[:, 0, :, 0] = (np.arange(n) // 16).astype(np.uint8)[:, None]            # 1024 distinct images
    bc = WaveletBatchCodec(n, h, w)
    bc.upload(rgb)
    bc.encode_resident()
    rng = np.random.default_rng(2024)
    origins = np.stack([rng.integers(0, h - 224 + 1, n), rng.integers(0, w - 224 + 1, n)], axis=1)
    windows = [("w224_s%d" % s, origins // s, (224 // s, 224 // s), s) for s in (1, 2, 4, 8)]
    res["batch_shape"] = [n, h, w]
    resident(bc, windows, args.reps, res, "batch")
    bc.close()
    res["card_after"] = card()

    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    ok = all(v for k, v in res.items() if "_check_" in k)
    if not ok:
        sys.exit("a check failed: %s" % {k: v for k, v in res.items() if "_check_" in k})


if __name__ == "__main__":
    main()
