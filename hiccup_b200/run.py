"""File-level driver, drop-in for reference hiccup/run.py:13-43 (the caller of the hot path; SURVEY 8(f)
rank 1) plus a directory mode that feeds the batched GPU path.

    compress(path, output, style)      run.py:18-29   image file -> <output>/<name>.<STYLE>-hic
    decompress(path)                   run.py:32-43   .hic file -> pixels (the reference shows them in a window;
                                                       here they are returned, and written with `save=`);
                                                       thumbnail=True: the 1/8-scale preview of a DCT-mode file instead;
                                                       region=(top, left, height, width): that window of it instead;
                                                       scale=2 or 4: its 1/2- or 1/4-scale image instead
    compress_many(paths, output, ...)  additive: same-shaped images are encoded as one GPU batch and their files
                                       written by the library's host threads (batch.write_files)
    decompress_many(paths, ...)        additive: same-shaped `.hic` files are read and decoded as one GPU batch

Like the reference, `cv2.imread` delivers BGR and the codec treats channel 0 as R (run.py:19), so files
are interchangeable with the reference's in both directions.  Command line: python -m hiccup_b200.run
-c IMG... | -d HIC... [-t | --region T,L,H,W | --scale 2|4] [-s JPEG|HIC] [-o OUT] [-r], the subset of bin/belch.py:26-49 that does not need a display.
"""
import argparse
import collections
import os

import numpy as np

from hiccup_b200 import _lib, codec, compression, hicimage, model


def img_name(path, c):
    return os.path.split(path)[-1] + ".%s-hic" % c.value


def _read(path):
    import cv2
    rgb = cv2.imread(path)
    if rgb is None:
        raise RuntimeError("cannot read image %r" % (path,))
    return rgb


def compress(path, output, c=model.Compression.JPEG, restarts=False):
    """restarts=True appends restart records to the file (an extension entry the reference's reader ignores;
    this package's decoder then skips the synchronisation passes of the Huffman decode)."""
    rgb = _read(path)
    if c == model.Compression.JPEG:
        hi = codec.jpeg_encode(compression.jpeg_compression(rgb), restarts=restarts)
    elif c == model.Compression.HIC:
        hi = codec.wavelet_encode(compression.wavelet_compression(rgb), restarts=restarts)
    else:
        raise RuntimeError("Unknown compression type")
    out = os.path.join(output, img_name(path, c))
    hi.write_file(out)
    return out


class _Output(collections.namedtuple("_Output", "suffix reduced decode decode_batch window")):
    """What decompress() and decompress_many() make of each file: the PNG name suffix, the name of the reduced decode
    (None for the full one), the single-file decode (HicImage -> pixels), the batch decode ((codec, EncodedStreams) ->
    pixels) and the region's ((top, left), (height, width)) or None."""

    def check(self, path, mode, shape=None):
        """NotImplementedError for a wavelet file asked for a reduced decode; ValueError for an image of `shape` that
        does not hold the window."""
        if self.reduced and mode != model.Compression.JPEG:
            raise NotImplementedError("%s is a wavelet (HIC) file: %s works on DCT-mode (JPEG) files" % (path, self.reduced))
        if self.window is not None and shape is not None:
            _lib.region_origins(*shape, [self.window[0]], self.window[1])


def _decode(hi):
    if hi.hic_type == model.Compression.JPEG:
        return compression.jpeg_decompression(codec.jpeg_decode(hi))
    if hi.hic_type == model.Compression.HIC:
        return compression.wavelet_decompression(codec.wavelet_decode(hi))
    raise RuntimeError("Unknown compression type")


def _output(thumbnail=False, region=None, scale=None):
    """The _Output for these options; ValueError for a malformed region, a scale other than 2 or 4, or more than one
    of thumbnail, region and scale."""
    if bool(thumbnail) + (region is not None) + (scale is not None) > 1:
        raise ValueError("thumbnail, region and scale do not go together: choose one")
    if region is not None:
        r = tuple(region)
        if len(r) != 4 or not all(isinstance(v, (int, np.integer)) for v in r):
            raise ValueError("region must be four integers (top, left, height, width), got %r" % (region,))
        top, left, height, width = (int(v) for v in r)
        origin = np.array([[top, left]], np.int32)
        return _Output(".region.png", "region decode", lambda hi: codec.jpeg_region(hi, top, left, height, width),
                       lambda bc, enc: bc.decode_regions(enc, np.tile(origin, (bc.n, 1)), (height, width)),
                       ((top, left), (height, width)))
    if scale is not None:
        scale = _lib.scale_arg(scale)
        return _Output(".s%d.png" % scale, "scaled decode", lambda hi: codec.jpeg_scaled(hi, scale),
                       lambda bc, enc: bc.decode_scaled(enc, scale), None)
    if thumbnail:
        return _Output(".thumb.png", "thumbnail decode", codec.jpeg_thumbnail, lambda bc, enc: bc.thumbnails(enc), None)
    return _Output(".png", None, _decode, lambda bc, enc: bc.decode(enc), None)


def decompress(path, save=None, thumbnail=False, region=None, scale=None):
    """thumbnail=True: the 1/8-scale preview (one pixel per 8x8 tile of the decoded image) of a DCT-mode file from its DC streams alone
    (codec.jpeg_thumbnail); a wavelet file raises NotImplementedError.  region=(top, left, height, width): that window
    of the decoded image at full resolution (codec.jpeg_region); a wavelet file raises NotImplementedError and a window
    the image does not hold ValueError, before anything is decoded or written.  scale=2 or 4: the 1/2- or 1/4-scale
    image of a DCT-mode file (codec.jpeg_scaled); a wavelet file raises NotImplementedError and another scale
    ValueError, before anything is decoded or written."""
    what = _output(thumbnail, region, scale)
    hi = hicimage.HicImage.from_file(path)
    what.check(path, hi.hic_type)
    rgb = what.decode(hi)
    if save is not None:
        import cv2
        cv2.imwrite(save, rgb)
    return rgb


def compress_many(paths, output, c=model.Compression.JPEG, max_batch=256, restarts=False):
    """Encode many files; images of one shape go through the batched codec together (one launch of
    every kernel per group) and every `.hic` file equals what compress() writes for it."""
    import numpy as np
    from hiccup_b200.batch import DctBatchCodec, WaveletBatchCodec
    groups = {}
    for p in paths:
        rgb = _read(p)
        groups.setdefault(rgb.shape, []).append((p, rgb))
    written = []
    for shape, items in groups.items():
        h, w = shape[:2]
        for a in range(0, len(items), max_batch):
            part = items[a:a + max_batch]
            cls = DctBatchCodec if c == model.Compression.JPEG else WaveletBatchCodec
            bc = cls(len(part), h, w)
            try:
                enc = bc.encode(np.stack([rgb for _, rgb in part]))
                outs = [os.path.join(output, img_name(p, c)) for p, _ in part]
                if restarts:
                    for out, hi in zip(outs, bc.hic_images(enc)):
                        codec.add_restart_records(hi).write_file(out)
                else:
                    bc.write_files(enc, outs)
                written += outs
            finally:
                bc.close()
    return written


def _peek(raw):
    """(mode, (h, w) of the image) of a `.hic` file's bytes, without touching its tables."""
    entries = hicimage.loads(raw)
    mode = model.Compression(hicimage.PlainStringP.from_bytes(entries[0]).payload)
    if mode == model.Compression.JPEG:
        shape = tuple(int(v) for v in hicimage.TupP.from_bytes(entries[19]).numbers)
    else:
        big = tuple(int(v) for v in hicimage.TupP.from_bytes(entries[14]).numbers)      # cD_1: half the image each way
        shape = (2 * big[0], 2 * big[1])
    return mode, shape


def decompress_many(paths, save_dir=None, max_batch=256, thumbnail=False, region=None, scale=None):
    """Decode many `.hic` files; files of one mode and image shape go through the batched codec together.  Returns the
    pixel arrays in the order of `paths` (equal to what decompress() returns for each); save_dir: also write them as PNG
    (<name>.png, or <name>.thumb.png for thumbnails).  thumbnail=True: the previews of DCT-mode files
    (DctBatchCodec.thumbnails); a wavelet file among them raises NotImplementedError before anything is decoded.
    region=(top, left, height, width): that window of every file (DctBatchCodec.decode_regions, <name>.region.png); a
    wavelet file, or a file whose image does not hold the window, raises before anything is decoded or written.
    scale=2 or 4: the 1/2- or 1/4-scale image of every file (DctBatchCodec.decode_scaled, <name>.s2.png / <name>.s4.png);
    a wavelet file or another scale raises before anything is decoded or written."""
    from hiccup_b200.batch import DctBatchCodec, WaveletBatchCodec
    what = _output(thumbnail, region, scale)
    groups, out = {}, [None] * len(paths)
    for i, p in enumerate(paths):
        with open(p, "rb") as f:
            raw = f.read()
        key = _peek(raw)
        what.check(p, *key)
        groups.setdefault(key, []).append((i, raw))
    for (mode, (h, w)), items in groups.items():
        cls = DctBatchCodec if mode == model.Compression.JPEG else WaveletBatchCodec
        for a in range(0, len(items), max_batch):
            part = items[a:a + max_batch]
            bc = cls(len(part), h, w)
            try:
                pixels = what.decode_batch(bc, bc.streams_from_files([raw for _, raw in part]))
                for (i, _), rgb in zip(part, pixels):
                    out[i] = rgb.copy()
            finally:
                bc.close()
    if save_dir is not None:
        import cv2
        for p, rgb in zip(paths, out):
            cv2.imwrite(os.path.join(save_dir, _png_name(p, what)), rgb)
    return out


def _png_name(path, what):
    return os.path.split(path)[-1] + what.suffix


def _parse_region(text):
    parts = text.split(",")
    try:
        vals = tuple(int(v) for v in parts)
    except ValueError:
        vals = ()
    if len(vals) != 4:
        raise argparse.ArgumentTypeError("expected TOP,LEFT,HEIGHT,WIDTH (four integers), got %r" % (text,))
    return vals


def main(argv=None):
    ap = argparse.ArgumentParser(description="hiccup image compression on the GPU (no GUI)")
    ap.add_argument("--compress", "-c", metavar="IMG_PATH", nargs="+")
    ap.add_argument("--decompress", "-d", metavar="HIC", nargs="+")
    ap.add_argument("--compression", "-s", metavar="STYLE", default=model.Compression.HIC.value,
                    choices=[model.Compression.HIC.value, model.Compression.JPEG.value])
    ap.add_argument("--output", "-o", metavar="OUT", default=".")
    ap.add_argument("--restarts", "-r", action="store_true",
                    help="append restart records to the .hic files (ignored by the reference's reader; faster decode here)")
    ap.add_argument("--thumbnail", "-t", action="store_true",
                    help="with -d: write the 1/8-scale preview of each DCT-mode file (<name>.thumb.png) from its DC streams alone")
    ap.add_argument("--region", metavar="TOP,LEFT,HEIGHT,WIDTH", type=_parse_region,
                    help="with -d: write that window of each DCT-mode file's decoded image (<name>.region.png) at full resolution")
    ap.add_argument("--scale", type=int, choices=(2, 4),
                    help="with -d: write the 1/2- or 1/4-scale image of each DCT-mode file (<name>.s2.png / <name>.s4.png)")
    args = ap.parse_args(argv)
    if (args.thumbnail or args.region is not None or args.scale is not None) and not args.decompress:
        ap.error("-t/--thumbnail, --region and --scale go with -d/--decompress")
    try:
        what = _output(args.thumbnail, args.region, args.scale)
    except ValueError as e:
        ap.error(str(e))
    style = model.Compression(args.compression)
    if args.compress:
        for out in (compress_many(args.compress, args.output, style, restarts=args.restarts) if len(args.compress) > 1
                    else [compress(args.compress[0], args.output, style, restarts=args.restarts)]):
            print(out)
    elif args.decompress:
        extra = {k: v for k, v in (("region", args.region), ("scale", args.scale)) if v is not None}
        if len(args.decompress) > 1:
            decompress_many(args.decompress, save_dir=args.output, thumbnail=args.thumbnail, **extra)
        else:
            decompress(args.decompress[0], save=os.path.join(args.output, _png_name(args.decompress[0], what)),
                       thumbnail=args.thumbnail, **extra)
        for p in args.decompress:
            print(os.path.join(args.output, _png_name(p, what)))
    else:
        raise RuntimeError("Illegal state")


if __name__ == "__main__":
    main()
