"""Thumbnail decode against the full decode, on one GPU (development aid; bench.py is the contract).

    python tools/thumb_time.py [--reps 10] [--out profiles/r03_thumb_b200.json]

  C2 device-resident   DctBatchCodec(1024, 426, 640): decode_device() against thumbnails_device(), from the
                       encoder's own device output (CUDA events, after warm-up, the two alternating)
  C2 from .hic files   read_files() + decode() against read_files() + thumbnails() of the batch's 1024 files
                       (host clock: the calls end in a device synchronise)
  C5 one file          16384^2: codec.jpeg_decode + compression.jpeg_decompression against codec.jpeg_thumbnail
and, in a separate profiled pass, the kernels of thumbnails_device().  Checks the batch thumbnails of eight seeded
images against per-image codec.jpeg_thumbnail.  Prints and writes one JSON line with the card's name and power limit.
"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                 # the name still comes from the library below
        return {"query_error": repr(e)}


def event_ms(fn, reps):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def host_ms(fn, reps):
    out = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        out.append((time.perf_counter() - t) * 1e3)
    return statistics.median(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_thumb_b200.json"))
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
    res = {"tool": "thumb_time", "device": buf.value.decode(), "card": card(), "reps": args.reps}
    torch.cuda.init()

    # ---- C2: 1024 x 640x426, the benchmark's images (seeds 2000..) -------------------------------------------
    n, h, w = 1024, 426, 640
    base = bench.synthetic_batch(16, h, w, 2000)
    rgb = np.ascontiguousarray(base[np.arange(n) % 16])
    rgb[:, 0, :, 0] = (np.arange(n) // 16).astype(np.uint8)[:, None]            # 1024 distinct images
    bc = DctBatchCodec(n, h, w)
    bc.upload(rgb)
    enc = bc.encode_resident()
    res["c2_payload_bytes"] = int(enc.data.nbytes)
    res["c2_dc_payload_bits_share"] = float(np.asarray(enc.nbits, np.float64)[0::3].sum() / np.asarray(enc.nbits, np.float64).sum())
    for _ in range(3):
        bc.decode_device()
        bc.thumbnails_device()
    torch.cuda.synchronize()
    full, thumb = [], []
    for _ in range(3):                      # alternating windows
        full.append(event_ms(bc.decode_device, args.reps))
        thumb.append(event_ms(bc.thumbnails_device, args.reps))
    res["c2_resident_decode_ms"] = statistics.median(full)
    res["c2_resident_thumbnail_ms"] = statistics.median(thumb)
    res["c2_resident_windows_ms"] = {"decode": full, "thumbnail": thumb}
    _lib.profile_enable(True)
    _lib.profile_report()
    bc.thumbnails_device()
    _lib.sync()
    res["c2_thumbnail_kernels_ms"] = {k: round(v[0], 4) for k, v in sorted(_lib.profile_report().items(), key=lambda kv: -kv[1][0])}
    bc.decode_device()
    _lib.sync()
    res["c2_decode_kernels_ms"] = {k: round(v[0], 4) for k, v in sorted(_lib.profile_report().items(), key=lambda kv: -kv[1][0])}
    _lib.profile_enable(False)

    tmp = tempfile.mkdtemp(prefix="thumb_time_")
    try:
        paths = [os.path.join(tmp, "%04d.hic" % i) for i in range(n)]
        bc.write_files(enc, paths)
        res["c2_file_bytes"] = sum(os.path.getsize(p) for p in paths)
        out_full = np.empty(bc.out_shape, np.uint8)
        out_thumb = np.empty(bc.thumbnail_shape, np.uint8)
        for _ in range(2):
            bc.decode(bc.read_files(paths), out=out_full)
            bc.thumbnails(bc.read_files(paths), out=out_thumb)
        full, thumb = [], []
        for _ in range(3):
            full.append(host_ms(lambda: bc.decode(bc.read_files(paths), out=out_full), max(2, args.reps // 3)))
            thumb.append(host_ms(lambda: bc.thumbnails(bc.read_files(paths), out=out_thumb), max(2, args.reps // 3)))
        res["c2_files_decode_ms"] = statistics.median(full)
        res["c2_files_thumbnail_ms"] = statistics.median(thumb)
        res["c2_files_windows_ms"] = {"decode": full, "thumbnail": thumb}
        read = host_ms(lambda: bc.read_files(paths), 3)
        res["c2_files_read_ms"] = read
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    pick = [int(i) for i in np.random.default_rng(2024).choice(n, 8, replace=False)]
    got = bc.thumbnails(enc)
    res["c2_check_images"] = pick
    res["c2_check_equal"] = all(np.array_equal(got[i], codec.jpeg_thumbnail(hi)) for i, hi in zip(pick, bc.hic_images(enc, images=pick)))
    bc.close()
    del rgb, base

    # ---- C5: one 16384^2 file ------------------------------------------------------------------------------
    size = 16384
    hic = bands.encode_banded(bench_bands.big_synthetic(size), 1)
    for _ in range(2):
        compression.jpeg_decompression(codec.jpeg_decode(hic))
        codec.jpeg_thumbnail(hic)
    full, thumb = [], []
    for _ in range(3):
        full.append(host_ms(lambda: compression.jpeg_decompression(codec.jpeg_decode(hic)), 2))
        thumb.append(host_ms(lambda: codec.jpeg_thumbnail(hic), 2))
    res["c5_decode_ms"] = statistics.median(full)
    res["c5_thumbnail_ms"] = statistics.median(thumb)
    res["c5_windows_ms"] = {"decode": full, "thumbnail": thumb}
    _lib.profile_enable(True)
    _lib.profile_report()
    codec.jpeg_thumbnail(hic)
    _lib.sync()
    res["c5_thumbnail_kernels_ms"] = {k: round(v[0], 4) for k, v in sorted(_lib.profile_report().items(), key=lambda kv: -kv[1][0])}
    _lib.profile_enable(False)
    res["card_after"] = card()

    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    if not res["c2_check_equal"]:
        sys.exit("batch thumbnails differ from codec.jpeg_thumbnail")


if __name__ == "__main__":
    main()
