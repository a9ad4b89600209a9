"""Scaled decode (1/2 and 1/4) against the full decode, on one GPU (development aid; bench.py is the contract).

    python tools/scaled_time.py [--reps 10] [--out profiles/r05_scaled_b200.json]

  C2 device-resident   DctBatchCodec(1024, 426, 640): decode_device() against decode_scaled_device(2) and (4), from
                       the encoder's own device output (CUDA events, after warm-up, the three alternating); per-kernel
                       times of each in a separate profiled pass (K7 + fix-up + K8 against K7S + fix-up + K8S)
  C2 from .hic files   read_files() + decode() against read_files() + decode_scaled(2) and (4) of the batch's 1024
                       files (host clock: the calls end in a device synchronise)
  C5 one file          16384^2: codec.jpeg_decode + compression.jpeg_decompression against codec.jpeg_scaled(2), (4)
Checks that the device-resident scaled images equal the host-to-host ones.  Prints and writes one JSON line with the
card's name and power limit.
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

from region_time import kernels
from thumb_time import card, event_ms, host_ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_scaled_b200.json"))
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
    res = {"tool": "scaled_time", "device": buf.value.decode(), "card": card(), "reps": args.reps}
    torch.cuda.init()

    # ---- C2: 1024 x 640x426, the benchmark's images (seeds 2000..) ----------------------------------------------
    n, h, w = 1024, 426, 640
    base = bench.synthetic_batch(16, h, w, 2000)
    rgb = np.ascontiguousarray(base[np.arange(n) % 16])
    rgb[:, 0, :, 0] = (np.arange(n) // 16).astype(np.uint8)[:, None]            # 1024 distinct images
    bc = DctBatchCodec(n, h, w)
    bc.upload(rgb)
    enc = bc.encode_resident()
    res["c2_blocks"] = int(n * bc.g.blocks_per_image)
    res["c2_out_bytes"] = {"full": int(np.prod(bc.out_shape)), "s2": int(np.prod(bc.scaled_shape(2))),
                           "s4": int(np.prod(bc.scaled_shape(4)))}
    calls = {"decode": bc.decode_device, "s2": lambda: bc.decode_scaled_device(2), "s4": lambda: bc.decode_scaled_device(4)}
    for _ in range(3):
        for fn in calls.values():
            fn()
    torch.cuda.synchronize()
    wins = {k: [] for k in calls}
    for _ in range(3):                      # alternating windows
        for k, fn in calls.items():
            wins[k].append(event_ms(fn, args.reps))
    res["c2_resident_ms"] = {k: statistics.median(v) for k, v in wins.items()}
    res["c2_resident_windows_ms"] = wins
    res["c2_kernels_ms"] = {k: kernels(fn, args.reps) for k, fn in calls.items()}
    check = True
    for s in (2, 4):
        bc.decode_scaled_device(s)
        dev = bc.fetch_scaled().copy()
        check &= bool(np.array_equal(dev, bc.decode_scaled(enc, s)))
    res["c2_check_equal"] = check

    tmp = tempfile.mkdtemp(prefix="scaled_time_")
    try:
        paths = [os.path.join(tmp, "%04d.hic" % i) for i in range(n)]
        bc.write_files(enc, paths)
        outs = {"decode": np.empty(bc.out_shape, np.uint8), 2: np.empty(bc.scaled_shape(2), np.uint8),
                4: np.empty(bc.scaled_shape(4), np.uint8)}
        calls = {"decode": lambda: bc.decode(bc.read_files(paths), out=outs["decode"]),
                 "s2": lambda: bc.decode_scaled(bc.read_files(paths), 2, out=outs[2]),
                 "s4": lambda: bc.decode_scaled(bc.read_files(paths), 4, out=outs[4])}
        for _ in range(2):
            for fn in calls.values():
                fn()
        wins = {k: [] for k in calls}
        for _ in range(3):
            for k, fn in calls.items():
                wins[k].append(host_ms(fn, max(2, args.reps // 3)))
        res["c2_files_ms"] = {k: statistics.median(v) for k, v in wins.items()}
        res["c2_files_windows_ms"] = wins
        res["c2_files_read_ms"] = host_ms(lambda: bc.read_files(paths), 3)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    bc.close()
    del rgb, base

    # ---- C5: one 16384^2 file -------------------------------------------------------------------------------------
    size = 16384
    hic = bands.encode_banded(bench_bands.big_synthetic(size), 1)
    calls = {"decode": lambda: compression.jpeg_decompression(codec.jpeg_decode(hic)),
             "s2": lambda: codec.jpeg_scaled(hic, 2), "s4": lambda: codec.jpeg_scaled(hic, 4)}
    for _ in range(2):
        for fn in calls.values():
            fn()
    wins = {k: [] for k in calls}
    for _ in range(3):
        for k, fn in calls.items():
            wins[k].append(host_ms(fn, 2))
    res["c5_ms"] = {k: statistics.median(v) for k, v in wins.items()}
    res["c5_windows_ms"] = wins
    res["c5_scaled_kernels_ms"] = {"s2": kernels(calls["s2"], 2), "s4": kernels(calls["s4"], 2)}
    res["card_after"] = card()

    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    if not res["c2_check_equal"]:
        sys.exit("device-resident scaled decode differs from the host-to-host one")


if __name__ == "__main__":
    main()
