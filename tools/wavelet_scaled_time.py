"""Wavelet scaled decode (1/2, 1/4, 1/8) against the full decode, on one GPU (development aid; bench.py is the contract).

    python tools/wavelet_scaled_time.py [--reps 10] [--out profiles/r07_wavelet_scaled_b200.json]

  C4 device-resident     WaveletBatchCodec(1, 4320, 7680), the benchmark's image: decode_device() against
                         decode_scaled_device(2), (4), (8) from the encoder's own device output (CUDA events, after
                         warm-up, alternating; medians of three windows); per-kernel times in a separate profiled pass
  transform only         on the decoded stream the codec holds: K10 (hic_wavelet_inverse) against
                         hic_wavelet_scaled_general at the default settings, per scale
  batch device-resident  the same for WaveletBatchCodec(1024, 432, 640) (C2's width, the height rounded up to a
                         multiple of 8)
  C4 from its .hic file  codec.wavelet_decode + compression.wavelet_decompression against codec.wavelet_scaled(s) (host
                         clock: the calls end in a device synchronise)
Checks that the device-resident scaled images equal the host-to-host ones and the transform-only ones.  Prints and writes one JSON line with the card's name, power limit and max SM clock.
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
from thumb_time import card, event_ms, host_ms

SCALES = (2, 4, 8)


def alternate(calls, reps):
    """Medians of three alternating event-timed windows per call (after one warm-up pass of each)."""
    import torch
    for fn in calls.values():
        fn()
    torch.cuda.synchronize()
    wins = {k: [] for k in calls}
    for _ in range(3):
        for k, fn in calls.items():
            wins[k].append(event_ms(fn, reps))
    return {k: statistics.median(v) for k, v in wins.items()}, wins


def resident(bc, enc, reps, res, tag):
    """decode_device against decode_scaled_device(s), then the transform stage alone: K10 against the scaled kernels."""
    from hiccup_b200 import _lib
    lib = bc.lib
    calls = {"decode": bc.decode_device}
    calls.update({"s%d" % s: (lambda s=s: bc.decode_scaled_device(s)) for s in SCALES})
    res[tag + "_resident_ms"], res[tag + "_resident_windows_ms"] = alternate(calls, reps)
    res[tag + "_kernels_ms"] = {k: kernels(fn, reps) for k, fn in calls.items()}
    check_dev = True
    host = {}
    for s in SCALES:
        bc.decode_scaled_device(s)
        host[s] = bc.fetch_scaled().copy()
    for s in SCALES:
        check_dev &= bool(np.array_equal(host[s], bc.decode_scaled(enc, s)))
    res[tag + "_check_resident_equals_host"] = check_dev

    # the transform stage alone on the stream decode_scaled left in d_coef_dec
    n, h, w = bc.n, bc.h, bc.w
    work = _lib.DeviceBuffer(_lib.wavelet_work_bytes(n, h, w))
    outs = {s: _lib.DeviceBuffer(n * (h // s) * (w // s) * 3) for s in SCALES}
    params = _lib.WaveletParams()
    params.levels, params.multiplier, params.threshold, params.threshold_index = 3, 1.0, 0.0, -1
    pref = ctypes.byref(params)
    full = _lib.DeviceBuffer(n * h * w * 3)
    calls = {"k10": lambda: _lib.check(lib.hic_wavelet_inverse(bc.d_coef_dec.ptr, n, h, w, full.ptr, None))}
    for s in SCALES:
        calls["general_s%d" % s] = lambda s=s: _lib.check(lib.hic_wavelet_scaled_general(bc.d_coef_dec.ptr, n, h, w, pref, s, work.ptr,
                                                                                         outs[s].ptr, None))
    res[tag + "_transform_ms"], res[tag + "_transform_windows_ms"] = alternate(calls, reps)
    res[tag + "_transform_kernels_ms"] = {k: kernels(fn, reps) for k, fn in calls.items()}
    agree = True
    for s in SCALES:
        count = n * (h // s) * (w // s) * 3
        calls["general_s%d" % s]()
        agree &= bool(np.array_equal(outs[s].download(np.uint8, count).reshape(host[s].shape), host[s]))
    res[tag + "_check_transform_equals_resident"] = agree
    for b in [work, full] + list(outs.values()):
        b.free()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_wavelet_scaled_b200.json"))
    args = ap.parse_args()
    import torch
    import bench
    from hiccup_b200 import _lib, codec, compression
    from hiccup_b200.batch import WaveletBatchCodec
    _lib.require_device()
    buf = ctypes.create_string_buffer(256)
    _lib.check(_lib.load().hic_device_name(buf, len(buf)))
    res = {"tool": "wavelet_scaled_time", "device": buf.value.decode(), "card": card(), "reps": args.reps}
    torch.cuda.init()

    # ---- C4: one 7680x4320 image, the benchmark's (seed 2000) -------------------------------------------------------
    h, w = 4320, 7680
    rgb = bench.synthetic_batch(1, h, w, 2000)
    bc = WaveletBatchCodec(1, h, w)
    bc.upload(rgb)
    enc = bc.encode_resident()
    hic = bc.hic_images(enc)[0]
    res["c4_out_bytes"] = {"full": int(np.prod(bc.out_shape)), **{"s%d" % s: int(np.prod(bc.scaled_shape(s))) for s in SCALES}}
    resident(bc, enc, args.reps, res, "c4")

    calls = {"decode": lambda: compression.wavelet_decompression(codec.wavelet_decode(hic))}
    calls.update({"s%d" % s: (lambda s=s: codec.wavelet_scaled(hic, s)) for s in SCALES})
    for fn in calls.values():
        fn()
    wins = {k: [] for k in calls}
    for _ in range(3):
        for k, fn in calls.items():
            wins[k].append(host_ms(fn, max(2, args.reps // 3)))
    res["c4_file_ms"] = {k: statistics.median(v) for k, v in wins.items()}
    res["c4_file_windows_ms"] = wins
    res["c4_file_kernels_ms"] = {k: kernels(fn, 2) for k, fn in calls.items()}
    checks = []
    for s in SCALES:
        bc.decode_scaled_device(s)
        checks.append(bool(np.array_equal(bc.fetch_scaled()[0], codec.wavelet_scaled(hic, s))))
    res["c4_check_file_equals_resident"] = all(checks)
    bc.close()
    del rgb

    # ---- a batch: 1024 x 432x640 ---------------------------------------------------------------------------------------
    n, h, w = 1024, 432, 640
    base = bench.synthetic_batch(16, h, w, 2000)
    rgb = np.ascontiguousarray(base[np.arange(n) % 16])
    rgb[:, 0, :, 0] = (np.arange(n) // 16).astype(np.uint8)[:, None]            # 1024 distinct images
    bc = WaveletBatchCodec(n, h, w)
    bc.upload(rgb)
    enc = bc.encode_resident()
    res["batch_shape"] = [n, h, w]
    resident(bc, enc, args.reps, res, "batch")
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
