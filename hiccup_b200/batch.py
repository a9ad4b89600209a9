"""Batched, device-resident pipelines (additive entry points: the reference API is one image per
call, SURVEY section 8(b)).

    codec = DctBatchCodec(n, h, w)         # or WaveletBatchCodec(n, h, w)
    enc = codec.encode(rgb_batch)          # host uint8 (n, h, w, 3) -> EncodedStreams (tables + framed bits)
    rgb = codec.decode(enc)                # -> host uint8 (n, out_h, out_w, 3)
    images = codec.hic_images(enc)         # -> list of HicImage, byte-identical to the reference's

All buffers and both entropy plans are allocated once for the shape; a step launches the same
kernels as the single-image drop-in functions (compression.py / codec.py / wavelet.py), just over n
images.  Host-side results are views of page-locked staging owned by the codec (valid until the next
call of the same method).
"""
import functools
import os

import numpy as np

from hiccup_b200 import _compat, _lib, entropy, hicimage, model


class _BatchCodec:
    """Shared plumbing: buffers, entropy plans, pinned staging.  Subclasses provide the transform."""

    def __init__(self, n, h, w, layout, coef_bytes, out_hw, value_bins, device, stream, device_codes):
        self.lib = _lib.load()
        self.n, self.h, self.w = int(n), int(h), int(w)
        self.stream = stream
        self.device_codes = bool(device_codes) and value_bins <= 8192      # E2 on the GPU (same codes, no PCIe)
        self.layout = layout
        self.out_h, self.out_w = out_hw
        self.d_rgb = _lib.DeviceBuffer(self.n * h * w * 3)
        self.d_coef = _lib.DeviceBuffer(coef_bytes)
        self.d_coef_dec = _lib.DeviceBuffer(coef_bytes)
        self.d_out = _lib.DeviceBuffer(self.n * self.out_h * self.out_w * 3)
        self.encoder = entropy.EntropyEncoder(self.layout, value_bins)
        self.decoder = entropy.EntropyDecoder(self.layout)
        self._buffers = [self.d_rgb, self.d_coef, self.d_coef_dec, self.d_out]
        self._reduced = {}
        # page-locked staging for the host-to-host entry points (grown on demand, reused every call)
        self._h_data = None
        self._h_out = None
        self._h_tab = None
        self._h_tab_mem = []

    # ---- sizes -------------------------------------------------------------------------------
    @property
    def pixels(self):
        return self.n * self.h * self.w

    @property
    def out_shape(self):
        return (self.n, self.out_h, self.out_w, 3)

    # ---- `.hic` files of a batch -----------------------------------------------------------------
    def hic_files(self, enc, images=None, threads=None, reuse=False):
        """The bytes of every image's `.hic` file (what HicImage.write_file dumps: pickle.dumps(hi.byte_stream()) for hi in
        hic_images(enc)), written for the whole batch by host threads of the library (hic_hicfile_pack_files) instead of
        one Python object per table row; files the library declines, or all of them where it did not calibrate against
        this environment's pickle, come from hic_images().  Returns a list of bytes-like objects.  reuse=True writes into
        a buffer the codec keeps (like its other staging: the result is valid until the next such call)."""
        import pickle
        images = list(range(self.n) if images is None else images)
        nat = hicimage._native()
        res = None
        if images and nat.files_ok:
            stream_of, modes, lead, trail = self._file_plan(images)
            res = nat.pack_files(_compat.wire_tuple_class(), enc.index, enc.symbols, enc.packed, enc.data, enc.byte_off, enc.byte_len,
                                 stream_of, modes, lead, trail, threads, reuse=self.__dict__.setdefault("_files_keep", {}) if reuse else None)
        out = []
        for j, i in enumerate(images):
            if res is not None and int(res[2][j]):
                a = int(res[1][j])
                out.append(memoryview(res[0])[a:a + int(res[2][j])])
            else:
                out.append(pickle.dumps(self.hic_images(enc, images=[i])[0].byte_stream()))
        return out

    def streams_from_files(self, files, threads=None):
        """The reverse of hic_files(): n bytes-like `.hic` files of this codec's mode and image shape -> the EncodedStreams
        decode() takes.  Canonical files (what pickle protocol 4 / 5 writes: the reference's and this package's) are walked
        by host threads of the library (hic_hicfile_scan_files / _parse_files); anything else goes through HicImage.from_bytes.
        Files of another mode or shape raise ValueError."""
        files = list(files)
        if len(files) != self.n:
            raise ValueError("%d files for a codec of %d images" % (len(files), self.n))
        stream_of, _, lead, trail = self._file_plan(list(range(self.n)))
        n_streams = 9 * self.n
        res = hicimage._native().parse_files(files, stream_of, n_streams, len(trail), threads) if self.n else None
        if res is not None:
            index, symbols, packed, data, byte_off, byte_len, nbits, leads, trails = res
            if all(l == lead for l in leads) and all(t == trail for t in trails):
                return entropy.EncodedStreams(self.layout, index, None, nbits, byte_off, byte_len, symbols, packed, data)
        # the tolerant path: any pickle protocol, any spelling of the shapes
        from hiccup_b200 import codec as codec_mod
        rows = np.zeros(n_streams, np.uint32)
        per_stream, framed = [None] * n_streams, [b""] * n_streams
        tables = stream_of.shape[1]
        for i, f in enumerate(files):
            hi = hicimage.HicImage.from_bytes(hicimage.loads(bytes(f)))
            if getattr(hi.hic_type, "value", hi.hic_type).encode() != lead or [tuple(int(v) for v in p.numbers) for p in hi.payloads[2 * tables:2 * tables + 2]] != \
                    [tuple(int(v) for v in hicimage.TupP.from_bytes(t).numbers) for t in trail]:
                raise ValueError("file %d is not a %s file of this codec's image shape" % (i, lead.decode()))
            for k in range(tables):
                s = int(stream_of[i, k])
                r, sym, lens, codes = codec_mod._tables_to_arrays([hi.payloads[k]])
                rows[s] = r[0]
                per_stream[s] = (sym, (lens.astype(np.uint64) << np.uint64(58)) | (codes & entropy.CODE_MASK))
                framed[s] = bytes(hi.payloads[tables + k].byte_stream)
        index = np.zeros((n_streams, 2), np.uint32)
        index[:, 1] = rows
        index[1:, 0] = np.cumsum(rows[:-1], dtype=np.uint64).astype(np.uint32)
        present = [p for p in per_stream if p is not None]
        symbols = np.concatenate([p[0] for p in present]).astype(np.int32) if present else np.zeros(0, np.int32)
        packed = np.concatenate([p[1] for p in present]).astype(np.uint64) if present else np.zeros(0, np.uint64)
        byte_len = np.array([len(b) for b in framed], np.uint64)
        padded = (byte_len + np.uint64(3)) & ~np.uint64(3)
        byte_off = np.zeros(n_streams, np.uint64)
        byte_off[1:] = np.cumsum(padded[:-1])
        data = np.zeros(int(padded.sum()) + 16, np.uint8)
        for b, a in zip(framed, byte_off.tolist()):
            data[a:a + len(b)] = np.frombuffer(b, np.uint8)
        nbits = np.array([hicimage.iohelper.payload_bit_count(b) if b else 0 for b in framed], np.uint64)
        return entropy.EncodedStreams(self.layout, index, None, nbits, byte_off, byte_len, symbols, packed, data)

    def read_files(self, paths, threads=None):
        """streams_from_files() of files on disk."""
        files = []
        for path in paths:
            with open(path, "rb") as f:
                files.append(f.read())
        return self.streams_from_files(files, threads)

    def write_files(self, enc, paths, images=None, threads=None):
        """hic_files() to disk: paths[j] receives the file of images[j]."""
        files = self.hic_files(enc, images, threads, reuse=True)
        assert len(files) == len(paths)
        for path, b in zip(paths, files):
            with open(path, "wb") as f:
                f.write(b)

    # ---- transform hooks ---------------------------------------------------------------------
    def _forward(self):
        raise NotImplementedError

    def _inverse(self):
        raise NotImplementedError

    # ---- device-resident steps ---------------------------------------------------------------
    def upload(self, rgb):
        rgb = np.ascontiguousarray(rgb, np.uint8)
        assert rgb.shape == (self.n, self.h, self.w, 3), rgb.shape
        self.d_rgb.upload(rgb, self.stream)

    def encode_device(self):
        """Transform, E1 (symbols + histograms), E2 (Huffman codes), E3 (bit packing); all in HBM."""
        st = self.stream
        self._forward()
        self.encoder.symbolize(self.d_coef.ptr, st)
        self.encoder.build_codes(st, on_device=self.device_codes)
        return self.encoder.pack(st)

    def decode_device(self):
        """D1-D3 and the inverse transform from the encoder's own device-resident output (tables
        and bits are handed over device-to-device)."""
        self._decode_from_encoder(self.d_coef_dec)
        self._inverse()

    def _decode_from_encoder(self, d_dst, dc_only=False):
        """D1-D3 of the encoder's own device-resident output (tables and bits are handed over device-to-device) into
        d_dst: the coefficient blocks, or with dc_only the DC streams alone, one value per block (EntropyDecoder.run_dc)."""
        st = self.stream
        enc = self.encoder
        d_index, d_row_sym, d_row_packed, _, _ = enc.device_tables()
        self.decoder.set_tables_device(d_index, d_row_sym, d_row_packed, enc.total_rows, st)
        run = self.decoder.run_dc if dc_only else self.decoder.run
        run(enc._out.ptr, enc.byte_off, enc.nbits, d_dst.ptr, st)

    def _decode_from_streams(self, enc, d_dst, dc_only=False):
        """D1-D3 of an EncodedStreams (its tables and bytes go up) into d_dst: the coefficient blocks, or with dc_only the
        DC streams alone, one value per block (only their tables and bytes go up; EntropyDecoder.decode_dc)."""
        if dc_only:
            self.decoder.decode_dc(*entropy.dc_streams_only(enc), d_dst.ptr, self.stream)
        else:
            self.decoder.decode_streams(enc, d_dst.ptr, self.stream)

    # ---- host-to-host entry points -----------------------------------------------------------
    def encode(self, rgb):
        self.upload(rgb)
        return self.encode_resident()

    def encode_resident(self):
        """Encode the batch already uploaded with upload(); returns the host-side EncodedStreams."""
        out = self.encode_device()
        enc = self.encoder
        nbytes = int(enc.total_bytes)
        if self._h_data is None or self._h_data.nbytes < nbytes:
            if self._h_data is not None:
                self._h_data.free()
            self._h_data = _lib.PinnedBuffer(nbytes + nbytes // 4 + 4096)
        data = out.download(np.uint8, nbytes, self.stream, out=self._h_data.array(np.uint8, nbytes))
        rows = int(enc.total_rows)
        if self._h_tab is None or self._h_tab[1].size < rows:
            for b in self._h_tab_mem:
                b.free()
            cap = rows + rows // 4 + 1024
            self._h_tab_mem = [_lib.PinnedBuffer(8 * enc.n_streams), _lib.PinnedBuffer(4 * cap), _lib.PinnedBuffer(8 * cap)]
            self._h_tab = (self._h_tab_mem[0].array(np.uint32), self._h_tab_mem[1].array(np.int32),
                           self._h_tab_mem[2].array(np.uint64))
        index, sym, packed = enc.tables_packed(self.stream, out=self._h_tab)
        self._after_encode()
        return entropy.EncodedStreams(self.layout, index, enc.nsym.copy(), enc.nbits.copy(),
                                      enc.byte_off.copy(), enc.byte_len.copy(), sym, packed, data)

    def download_payload_sized(self):
        """The device->host copies of encode_resident() without its kernels: as many payload and table bytes
        as the last real encode of this codec produced (PipelinedCodec's copy-only floor)."""
        enc = self.encoder
        nbytes = int(getattr(enc, "total_bytes", 0) or 0)
        if not nbytes or self._h_data is None or enc._out is None:
            raise RuntimeError("copy-only pass before any real encode of this codec")
        enc._out.download(np.uint8, nbytes, self.stream, out=self._h_data.array(np.uint8, nbytes))
        enc.tables_packed(self.stream, out=self._h_tab)

    def decode(self, enc, out=None):
        """out: optional preallocated uint8 array of out_shape (ideally page-locked) to receive the pixels."""
        self.decode_resident(enc)
        return self.fetch(out)

    def decode_resident(self, enc):
        """Entropy-decode and inverse-transform an EncodedStreams; the pixels stay on the device."""
        self._decode_from_streams(enc, self.d_coef_dec)
        self._inverse()

    def fetch(self, out=None):
        """Download the pixels of the last decode_resident()."""
        pixels, self._h_out = self._download(self.d_out, self.out_shape, out, self._h_out)
        self._after_decode()
        return pixels

    def _download(self, d_buf, shape, out, staging):
        """The uint8 array of `shape` at the start of d_buf, downloaded into `out` (a C-contiguous uint8 array of its
        size) or, without one, into `staging`, page-locked memory the caller keeps (made here when None).  Returns
        (the array, staging)."""
        count = int(np.prod(shape))
        if out is None:
            if staging is None:
                staging = _lib.PinnedBuffer(count)
            out = staging.array(np.uint8, count)
        else:
            assert out.dtype == np.uint8 and out.size == count and out.flags.c_contiguous
            out = out.reshape(-1)
        return d_buf.download(np.uint8, count, self.stream, out=out).reshape(shape), staging

    def _after_encode(self):
        pass

    def _after_decode(self):
        pass

    def _after_scaled(self):
        pass

    # ---- reduced outputs (thumbnails, regions, scaled images) ---------------------------------------------------------
    def _reduced_buffers(self, kind, key, sizes):
        """The buffers of reduced output `kind` for its parameters `key`.  Each kind keeps its own, made on first use (a
        codec that never asks for one pays nothing) and remade only when its key changes; sizes() gives (output shape,
        work bytes, tie capacity) for a new key."""
        r = self._reduced.get(kind)
        if r is not None and r.key == key:
            return r
        if r is not None:
            self._reduced.pop(kind).free()
        r = self._reduced[kind] = _ReducedOutput(key, *sizes())
        return r

    def _run_reduced(self, r, launch, enc=None, dc_only=False, d_src=None):
        """D1-D3 into d_src (default the coefficient buffer of decode_device) -- from the encoder's own device-resident
        output (decode_device's hand-over) or, given `enc`, from that EncodedStreams; all streams, or with dc_only the DC
        streams alone -- then launch(r), the kernels of reduced output r."""
        d_src = self.d_coef_dec if d_src is None else d_src
        if enc is None:
            self._decode_from_encoder(d_src, dc_only)
        else:
            self._decode_from_streams(enc, d_src, dc_only)
        launch(r)

    def _fetch_reduced(self, r, out):
        """Download reduced output r into `out` or, without one, into its page-locked staging."""
        pixels, r.h_out = self._download(r.d_out, r.shape, out, r.h_out)
        return pixels

    # ---- 1/scale images (codec.jpeg_scaled or codec.wavelet_scaled for the whole batch); the subclasses provide
    # scaled_shape(scale), _scaled_buffers(scale) and _scaled(r) ------------------------------------------------------
    def decode_scaled_device(self, scale):
        """D1-D3 from the encoder's own device-resident output (decode_device's hand-over), then the 1/scale images;
        they stay on the device (fetch_scaled)."""
        self._run_reduced(self._scaled_buffers(scale), self._scaled)

    def decode_scaled(self, enc, scale, out=None):
        """The 1/scale images of an EncodedStreams, host to host: image i equals codec.jpeg_scaled (scale 2 or 4) or
        codec.wavelet_scaled of its file, as the codec's mode.  out: optional preallocated uint8 array of
        scaled_shape(scale)."""
        self._run_reduced(self._scaled_buffers(scale), self._scaled, enc)
        return self.fetch_scaled(out)

    def fetch_scaled(self, out=None):
        """Download the images of the last decode_scaled() / decode_scaled_device() (and, in DCT mode, their tie
        statistics into scaled_stats)."""
        pixels = self._fetch_reduced(self._reduced["scaled"], out)
        self._after_scaled()
        return pixels

    # ---- windows: one height x width window per image of the full-resolution or 1/scale image (codec.jpeg_region or
    # codec.wavelet_region for the whole batch); the subclasses provide _region_buffers(origins, size, scale),
    # _region(origins, r) and _after_regions(r) --------------------------------------------------------------------------
    def decode_regions_device(self, origins, size, scale=1):
        """D1-D3 from the encoder's own device-resident output (decode_device's hand-over; in DCT mode DC-only at scale 8,
        as thumbnails_device), then the windows of size = (height, width) at origins ((n, 2) of (top, left), in the
        coordinates of the 1/scale image); they stay on the device (fetch_regions)."""
        origins, r, dc_only = self._region_buffers(origins, size, scale)
        self._run_reduced(r, functools.partial(self._region, origins), dc_only=dc_only)

    def decode_regions(self, enc, origins, size, out=None, scale=1):
        """Windows of an EncodedStreams, host to host: image i's window is decode(enc)[i, top:top+height,
        left:left+width] with (top, left) = origins[i] and (height, width) = size, bit for bit -- or the same window of
        decode_scaled(enc, scale)[i] (DCT mode: scale 2 or 4; wavelet mode: 2^k, 1 <= k <= levels), in DCT mode at
        scale 8 of thumbnails(enc)[i] (only the DC streams go up).  out: optional preallocated uint8 array of
        (n, height, width, 3)."""
        origins, r, dc_only = self._region_buffers(origins, size, scale)
        self._run_reduced(r, functools.partial(self._region, origins), enc, dc_only=dc_only)
        return self.fetch_regions(out)

    def fetch_regions(self, out=None):
        """Download the windows of the last decode_regions() / decode_regions_device() (and, in DCT mode, their tie
        statistics into region_stats; all zero at scale 8, which has no tie stage)."""
        r = self._reduced["region"]
        pixels = self._fetch_reduced(r, out)
        self._after_regions(r)
        return pixels

    def _after_regions(self, r):
        pass

    def _check_origin_count(self, origins):
        if origins.shape[0] != self.n:
            raise ValueError("%d origins for a batch of %d images" % (origins.shape[0], self.n))

    def close(self):
        for r in self._reduced.values():
            r.free()
        self._reduced = {}
        self.encoder.close()
        self.decoder.close()
        for b in self._buffers + [self._h_data, self._h_out] + self._h_tab_mem:
            if b is not None:
                b.free()
        self._buffers, self._h_data, self._h_out, self._h_tab, self._h_tab_mem = [], None, None, None, []


class _ReducedOutput:
    """The device buffers of one reduced output of a batch codec (thumbnails, regions or scaled images) for one key,
    its parameters: the kernels' work area and the output, plus the page-locked staging a fetch without `out` makes."""

    def __init__(self, key, shape, work_bytes, tie_capacity):
        self.key, self.shape, self.work_bytes, self.tie_capacity = key, shape, work_bytes, tie_capacity
        self.d_work = _lib.DeviceBuffer(work_bytes)
        self.d_out = _lib.DeviceBuffer(int(np.prod(shape)))
        self.h_out = None

    def free(self):
        for b in (self.d_work, self.d_out, self.h_out):
            if b is not None:
                b.free()


class DctBatchCodec(_BatchCodec):
    """DCT ("JPEG") mode: K1 + fix-up -> entropy stage -> K7 + fix-up, K8."""

    def __init__(self, n, h, w, value_bins=entropy.DEFAULT_VALUE_BINS, device=None, stream=None, device_codes=True):
        _lib.require_device()
        if device is not None:
            _lib.check(_lib.load().hic_set_device(int(device)))
        g = self.g = _lib.geometry(h, w)
        self.blocks = int(n) * g.blocks_per_image
        super().__init__(n, h, w, _lib.layout_dct(int(n), h, w), self.blocks * 128, (g.out_h, g.out_w), value_bins,
                         device, stream, device_codes)
        self.tie_capacity = _lib.tie_capacity(n, h, w)
        self.d_ties = _lib.DeviceBuffer(self.tie_capacity * _lib.TIE_RECORD_BYTES)
        self.d_stats = _lib.DeviceBuffer(4 * _lib.TIE_STATS)
        self.d_y = _lib.DeviceBuffer(self.n * h * w)
        self.d_cr = _lib.DeviceBuffer(self.n * g.hc * g.wc)
        self.d_cb = _lib.DeviceBuffer(self.n * g.hc * g.wc)
        self._buffers += [self.d_ties, self.d_stats, self.d_y, self.d_cr, self.d_cb]
        self.forward_stats = np.zeros(4, np.uint32)
        self.inverse_stats = np.zeros(4, np.uint32)

    def _forward(self):
        _lib.check(self.lib.hic_dct_forward(self.d_rgb.ptr, self.n, self.h, self.w, self.d_coef.ptr, self.d_ties.ptr,
                                            self.tie_capacity, self.d_stats.ptr, self.stream))

    def _inverse(self):
        _lib.check(self.lib.hic_dct_inverse(self.d_coef_dec.ptr, self.n, self.h, self.w, self.d_y.ptr, self.d_cr.ptr,
                                            self.d_cb.ptr, self.d_out.ptr, self.d_ties.ptr, self.blocks,
                                            self.d_stats.ptr, self.stream))

    def _after_encode(self):
        self.forward_stats = self.d_stats.download(np.uint32, _lib.TIE_STATS, self.stream)

    def _after_decode(self):
        self.inverse_stats = self.d_stats.download(np.uint32, _lib.TIE_STATS, self.stream)

    # ---- 1/8-scale thumbnails from the DC streams alone (codec.jpeg_thumbnail for the whole batch) ---------------
    @property
    def thumbnail_shape(self):
        th, tw = _lib.thumbnail_shape(self.h, self.w)
        return (self.n, th, tw, 3)

    def _thumbnail_buffers(self):
        """The work area holds the DC values, one int16 per block."""
        return self._reduced_buffers("thumbnail", None, lambda: (self.thumbnail_shape, 2 * self.blocks, 0))

    def _thumbnail(self, r):
        _lib.check(self.lib.hic_dct_thumbnail(r.d_work.ptr, self.n, self.h, self.w, r.d_out.ptr, self.stream))

    def thumbnails_device(self):
        """DC-only D1 + D3 and the thumbnail kernel from the encoder's own device-resident output (decode_device's
        hand-over); the thumbnails stay on the device (fetch_thumbnails)."""
        r = self._thumbnail_buffers()
        self._run_reduced(r, self._thumbnail, dc_only=True, d_src=r.d_work)

    def thumbnails(self, enc, out=None):
        """Thumbnails of an EncodedStreams (encode() or read_files() / streams_from_files()), host to host: only the
        DC streams' tables and bytes go up, n x th x tw x 3 comes down.  out: optional preallocated uint8 array of
        thumbnail_shape."""
        r = self._thumbnail_buffers()
        self._run_reduced(r, self._thumbnail, enc, dc_only=True, d_src=r.d_work)
        return self.fetch_thumbnails(out)

    def fetch_thumbnails(self, out=None):
        """Download the thumbnails of the last thumbnails() / thumbnails_device()."""
        return self._fetch_reduced(self._thumbnail_buffers(), out)

    # ---- regions: one height x width window per image, of the full-resolution image (codec.jpeg_region for the whole
    # batch) or of the 1/2-, 1/4- or 1/8-scale image (jpeg_region(..., scale)) ----------------------------------------
    def _region_buffers(self, origins, size, scale):
        """Check the scale and the windows (ValueError before any device work); returns the origins as (n, 2) int32, the
        buffers for their size and scale, and whether the decode is DC-only (scale 8, as thumbnails)."""
        scale = _lib.region_scale_arg(scale)
        origins = _lib.region_origins(self.h, self.w, origins, size, scale)
        self._check_origin_count(origins)
        rh, rw = int(size[0]), int(size[1])
        if scale == 1:
            sizes = lambda: _lib.region_sizes(self.n, self.h, self.w, rh, rw)
        else:
            sizes = lambda: _lib.scaled_region_sizes(self.n, self.h, self.w, scale, rh, rw)
        return origins, self._reduced_buffers("region", (rh, rw, scale), lambda: ((self.n, rh, rw, 3),) + sizes()), scale == 8

    def _region(self, origins, r):
        """The region kernels of r's scale on the decoded coefficients -- at scale 8 on the DC values, which the DC-only
        decode leaves in the coefficient buffer."""
        rh, rw, scale = r.key
        if scale == 1:
            _lib.check(self.lib.hic_dct_region(self.d_coef_dec.ptr, self.n, self.h, self.w, origins.ctypes.data, rh, rw,
                                               r.d_work.ptr, r.work_bytes, self.d_ties.ptr, r.tie_capacity, self.d_stats.ptr,
                                               r.d_out.ptr, self.stream))
        elif scale == 8:
            _lib.check(self.lib.hic_dct_thumbnail_region(self.d_coef_dec.ptr, self.n, self.h, self.w, origins.ctypes.data, rh,
                                                         rw, r.d_work.ptr, r.work_bytes, r.d_out.ptr, self.stream))
        else:
            _lib.check(self.lib.hic_dct_scaled_region(self.d_coef_dec.ptr, self.n, self.h, self.w, scale, origins.ctypes.data,
                                                      rh, rw, r.d_work.ptr, r.work_bytes, self.d_ties.ptr, r.tie_capacity,
                                                      self.d_stats.ptr, r.d_out.ptr, self.stream))

    def _after_regions(self, r):
        """The tie statistics of the windows into region_stats: all zero at scale 8, which has no tie stage."""
        if r.key[2] == 8:
            self.region_stats = np.zeros(_lib.TIE_STATS, np.uint32)
        else:
            self.region_stats = self.d_stats.download(np.uint32, _lib.TIE_STATS, self.stream)

    # ---- 1/2- and 1/4-scale images (codec.jpeg_scaled for the whole batch) ----------------------------------------
    def scaled_shape(self, scale):
        sh, sw = _lib.scaled_shape(self.h, self.w, _lib.scale_arg(scale))
        return (self.n, sh, sw, 3)

    def _scaled_buffers(self, scale):
        """Check the scale (ValueError before any device work); returns the buffers for it."""
        scale = _lib.scale_arg(scale)
        return self._reduced_buffers(
            "scaled", scale, lambda: (self.scaled_shape(scale),) + _lib.scaled_sizes(self.n, self.h, self.w, scale))

    def _scaled(self, r):
        _lib.check(self.lib.hic_dct_scaled(self.d_coef_dec.ptr, self.n, self.h, self.w, r.key, r.d_work.ptr, r.work_bytes,
                                           self.d_ties.ptr, r.tie_capacity, self.d_stats.ptr, r.d_out.ptr, self.stream))

    def _after_scaled(self):
        self.scaled_stats = self.d_stats.download(np.uint32, _lib.TIE_STATS, self.stream)

    def coefficients(self):
        """Download the quantised zigzag blocks of the last encode: (n, blocks_per_image, 64) int16."""
        c = self.d_coef.download(np.int16, self.blocks * 64, self.stream)
        return c.reshape(self.n, self.g.blocks_per_image, 64)

    def hic_images(self, enc, images=None):
        """Materialise the reference's container objects (codec.jpeg_encode's return value) per image
        (images: the indices wanted; default all)."""
        g = self.g
        out = []
        for i in (range(self.n) if images is None else images):
            tables, bits = [], []
            for kind in range(3):
                for c in range(3):
                    s = (i * 3 + c) * 3 + kind
                    sym, lens, codes = enc.stream_rows(s)
                    tables.append(hicimage.PayloadStringP.from_arrays(sym, lens, codes, kind == entropy.KIND_DC))
                    bits.append(hicimage.BitStringP.from_framed(enc.framed(s)))
            out.append(hicimage.HicImage.jpeg_image(tables + bits + [hicimage.TupP(g.h, g.w), hicimage.TupP(g.hc, g.wc)]))
        return out


    def _file_plan(self, images):
        """(stream_of [files][9], flag modes, lead entry, trail entries) of hic_files(): the file order of
        HicImage.jpeg_image -- tables then bit strings, each kind-major / channel-minor -- and the two shape payloads."""
        g = self.g
        stream_of = np.array([[(i * 3 + c) * 3 + kind for kind in range(3) for c in range(3)] for i in images], np.uint32).reshape(-1, 9)
        modes = [1 if kind == entropy.KIND_DC else 0 for kind in range(3) for _ in range(3)]
        return (stream_of, modes, hicimage.PlainStringP(model.Compression.JPEG.value).byte_stream,
                [hicimage.TupP(g.h, g.w).byte_stream, hicimage.TupP(g.hc, g.wc).byte_stream])


class WaveletBatchCodec(_BatchCodec):
    """Wavelet ("HIC") mode: K9 -> flat-mode entropy stage -> K10 at the default settings, the general
    level-by-level kernels (csrc/hic_wavelet_general.cu) at any other settings.py values, read when the codec
    is made.  To decode, h and w must be multiples of 2^levels (the reference's decoder needs exact halvings,
    codec.py:182-189)."""

    def __init__(self, n, h, w, value_bins=entropy.DEFAULT_VALUE_BINS, device=None, stream=None, device_codes=True):
        import ctypes
        from hiccup_b200 import settings, wavelet
        _lib.require_device()
        settings.check_wavelet_supported()
        if device is not None:
            _lib.check(_lib.load().hic_set_device(int(device)))
        self.general = not settings.wavelet_defaults()
        if self.general:
            g = self.g = _lib.wavelet_pyramid(h, w, settings.WAVELET_NUM_LEVELS)
        else:
            g = self.g = _lib.wavelet_geometry(h, w)
        self.params = wavelet._params(g)           # the scaled decode runs the general kernels at every setting
        self._params_ref = ctypes.byref(self.params)
        self.chan_elems = 64 * ((int(g.len) + 63) // 64)
        super().__init__(n, h, w, _lib.layout_flat(int(n), int(g.len)), 2 * self.chan_elems * 3 * int(n), (h, w),
                         value_bins, device, stream, device_codes)
        self.d_work = None             # the general kernels' work area; a default-settings codec makes it for a scaled decode
        if self.general:
            self._make_work()

    def _make_work(self):
        self.d_work = _lib.DeviceBuffer(_lib.wavelet_work_bytes(self.n, self.h, self.w))
        self._buffers.append(self.d_work)

    def _forward(self):
        if self.general:
            _lib.check(self.lib.hic_wavelet_forward_general(self.d_rgb.ptr, self.n, self.h, self.w, self._params_ref,
                                                            self.d_work.ptr, self.d_coef.ptr, self.stream))
        else:
            _lib.check(self.lib.hic_wavelet_forward(self.d_rgb.ptr, self.n, self.h, self.w, self.d_coef.ptr, self.stream))

    def _inverse(self):
        if self.general:
            _lib.check(self.lib.hic_wavelet_inverse_general(self.d_coef_dec.ptr, self.n, self.h, self.w, self._params_ref,
                                                            self.d_work.ptr, self.d_out.ptr, self.stream))
        else:
            _lib.check(self.lib.hic_wavelet_inverse(self.d_coef_dec.ptr, self.n, self.h, self.w, self.d_out.ptr, self.stream))

    # ---- 1/2- to 1/2^levels-scale images (codec.wavelet_scaled for the whole batch) --------------------------------
    def scaled_shape(self, scale):
        """(n, h / scale, w / scale, 3); ValueError for a scale other than 2^k, 1 <= k <= levels, or sides that are not
        multiples of 2^levels."""
        levels = int(getattr(self.g, "levels", 3))
        s = 1 << _lib.wavelet_scale_arg(scale, levels)
        if self.h % (1 << levels) or self.w % (1 << levels):
            raise ValueError("a scaled decode of %d levels needs sides that are multiples of %d (got %dx%d)"
                             % (levels, 1 << levels, self.h, self.w))
        return (self.n, self.h // s, self.w // s, 3)

    def _scaled_buffers(self, scale):
        """Check the scale (ValueError before any device work); returns the output buffers for it.  The work area is the
        codec's, kept across scales; a default-settings codec makes it with its first scaled decode."""
        shape = self.scaled_shape(scale)
        if self.d_work is None:
            self._make_work()
        return self._reduced_buffers("scaled", int(scale), lambda: (shape, 0, 0))

    def _scaled(self, r):
        _lib.check(self.lib.hic_wavelet_scaled_general(self.d_coef_dec.ptr, self.n, self.h, self.w, self._params_ref, r.key,
                                                       self.d_work.ptr, r.d_out.ptr, self.stream))

    # ---- windows of the full-resolution or 1/2- to 1/2^levels-scale image (codec.wavelet_region for the whole batch) ---
    def _region_buffers(self, origins, size, scale):
        """Check the scale and the windows (ValueError before any device work); returns the origins as (n, 2) int32, the
        buffers for their size and scale (the work area holds the origins alone) and False: the decode is never DC-only."""
        origins = _lib.wavelet_region_origins(self.h, self.w, self.params.levels, origins, size, scale)
        self._check_origin_count(origins)
        rh, rw = int(size[0]), int(size[1])
        return origins, self._reduced_buffers("region", (rh, rw, int(scale)), lambda: ((self.n, rh, rw, 3), origins.nbytes, 0)), False

    def _region(self, origins, r):
        rh, rw, scale = r.key
        _lib.check(self.lib.hic_wavelet_region(self.d_coef_dec.ptr, self.n, self.h, self.w, self._params_ref, scale,
                                               origins.ctypes.data, rh, rw, r.d_work.ptr, r.work_bytes, r.d_out.ptr, self.stream))

    def hic_images(self, enc, images=None):
        from hiccup_b200 import wavelet
        return [wavelet.encode_streams_to_hic(enc, self.g, image=i) for i in (range(self.n) if images is None else images)]

    def _file_plan(self, images):
        """wavelet_image's order: 3 value tables, 3 length tables, their bit strings, cA_L's and cD_1's shapes (codec.py:147-163);
        non-zero values are numpy scalars in the pickles, zero and the zero counts Python ints."""
        from hiccup_b200 import wavelet
        stream_of = np.array([[(i * 3 + c) * 3 + kind for kind in (entropy.KIND_VALUE, entropy.KIND_LENGTH) for c in range(3)]
                              for i in images], np.uint32).reshape(-1, 6)
        shapes = wavelet.band_shapes(self.g)
        return (stream_of, [2, 2, 2, 0, 0, 0], hicimage.PlainStringP(model.Compression.HIC.value).byte_stream,
                [hicimage.TupP(*shapes[0]).byte_stream, hicimage.TupP(*shapes[-1]).byte_stream])


class PipelinedCodec:
    """A big batch as a pipeline of chunks over a few concurrent slots (each slot = one codec on its own
    CUDA stream, driven by its own host thread): the host->device copy of one chunk, the kernels of
    another and the device->host copy of a third overlap, so the host-to-host rate approaches
    max(PCIe, kernels) instead of their sum.  Results are identical to the unchunked codecs (images are
    independent).

        pipe = PipelinedCodec(1024, 426, 640, chunk=128, slots=3)            # mode="dct" | "wavelet"
        pipe.round_trip(rgb, out, on_encoded=lambda first_image, enc: ...)  # enc: EncodedStreams of a chunk
    """

    def __init__(self, n, h, w, chunk=128, slots=3, mode="dct", device=None, blocking_sync=False, **kw):
        _lib.require_device()
        if device is not None:
            _lib.check(_lib.load().hic_set_device(int(device)))
        self.device = device
        # Host threads spin while they wait (the driver's default).  Blocking waits (hic_set_blocking_sync) were
        # measured and are opt-in: they cost 4 % on one GPU (27.0 -> 28.0 ms per C2 batch) and do not help when
        # four pipelines share a box (71.6 -> 83.7 ms per batch and rank: the host side of PCIe is the limit
        # there, not the cores).
        if blocking_sync or os.environ.get("HIC_BLOCKING_SYNC"):
            _lib.check(_lib.load().hic_set_blocking_sync(1))
        self.n, self.h, self.w = int(n), int(h), int(w)
        self.chunk = max(1, min(int(chunk), self.n))
        if self.n % self.chunk:
            raise ValueError("batch of %d is not a whole number of %d-image chunks" % (self.n, self.chunk))
        self.n_chunks = self.n // self.chunk
        self.slots = max(1, min(int(slots), self.n_chunks))
        cls = DctBatchCodec if mode == "dct" else WaveletBatchCodec
        self.streams = [_lib.stream_create() for _ in range(self.slots)]
        self.codecs = [cls(self.chunk, h, w, stream=st, **kw) for st in self.streams]
        self.out_shape = (self.n,) + self.codecs[0].out_shape[1:]

    def round_trip(self, rgb, out, on_encoded=None, repeat=1, trace=None, resident=False, from_device=True,
                   copy_only=False):
        """Encode then decode every chunk of `rgb` (n, h, w, 3) into `out` (out_shape); both should be
        page-locked for the copies to overlap.  `repeat` > 1 streams the same batch through that many
        times without draining the pipeline in between (a stream of batches).  Returns the compressed
        payload bytes of one pass.

        Two gates keep the slots out of lockstep: one chunk at a time owns the bulk host->device copy
        and one the bulk device->host copy, so copies queue first-in first-out at full PCIe rate while
        the other slots are in their kernel phases.

        `from_device`: decode each chunk from the compressed payload and code tables the encoder left on the
        device (they are downloaded to the host all the same -- they are a result of the call -- but not
        uploaded again); False sends the host copy back up, as decoding a file would.

        `resident`: skip the bulk copies (each slot re-encodes the chunk its device buffer already holds
        and leaves the pixels on the device) -- the device-resident rate of the same pipeline.

        `copy_only`: the same bulk copies, slot threads and gates with NO kernels (the payload-sized download
        uses the size of the slot's last real encode): what PCIe alone allows this call -- its floor.

        `trace`: optional list that receives (slot, visit, phase, t_begin, t_end) host timestamps of the
        phases as they already synchronise (no extra synchronisation is added)."""
        assert rgb.shape == (self.n, self.h, self.w, 3) and out.shape == self.out_shape
        total = repeat * self.n_chunks

        def tickets(slot):
            for v in range(slot, total, self.slots):
                c = v % self.n_chunks
                yield v, c * self.chunk, rgb[c * self.chunk:(c + 1) * self.chunk], out[c * self.chunk:(c + 1) * self.chunk], v < self.n_chunks

        payload, _ = self._run(tickets, on_encoded, trace, resident, from_device, copy_only)
        return payload

    def upload_resident(self, rgb):
        """Park the batch in the slots' device buffers (chunk c in slot c; needs slots == chunks)."""
        assert self.slots == self.n_chunks, "one slot per chunk"
        for c, codec in enumerate(self.codecs):
            codec.upload(rgb[c * self.chunk:(c + 1) * self.chunk])
            _lib.sync(codec.stream)

    def device_steps(self, repeat=1, threads=None):
        """`repeat` encode+decode passes over the batch parked by upload_resident(), everything in HBM: every
        slot runs its chunk's kernels on its own CUDA stream from its own host thread, so one chunk's
        latency-bound stretches (the serial heapq replays of the Huffman builder, the table builds, the
        stream scans) run under another chunk's bandwidth-bound kernels.  No host<->device traffic besides
        the few status words the C ABI reads back.  Results are what encode_device() / decode_device() of
        each slot's codec leave on the device.  threads: host threads to drive the slots with (default one per
        slot; fewer when several ranks share the box's cores -- a thread then takes its slots in turn)."""
        import threading
        assert self.slots == self.n_chunks, "one slot per chunk"
        errors = []
        n_threads = self.slots if not threads else max(1, min(int(threads), self.slots))

        def work(first):
            try:
                if self.device is not None:
                    _lib.check(_lib.load().hic_set_device(int(self.device)))
                mine = [self.codecs[s] for s in range(first, self.slots, n_threads)]
                for _ in range(repeat):
                    for codec in mine:
                        codec.encode_device()
                    for codec in mine:
                        codec.decode_device()
                for codec in mine:
                    _lib.sync(codec.stream)
            except Exception as e:
                errors.append(e)

        threads = [threading.Thread(target=work, args=(t,)) for t in range(n_threads)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errors:
            raise errors[0]

    def run_job(self, job, repeat=1, on_encoded=None, from_device=True, copy_only=False, trace=None):
        """This rank's share of a box-wide job (hiccup_b200/jobs.py): chunks of EVERY rank's batch are handed
        out from one shared ticket counter, so a GPU whose path to host memory is faster -- PCIe root ports
        and sockets are not symmetric on a multi-GPU box -- takes more of them, and the job ends when the
        counter runs out instead of when the slowest link has moved a fixed share.  Images are independent
        (by-image partition, no collective); every rank reads and writes the shared, page-locked host
        buffers of the job directly.  Returns (payload bytes this rank produced in the first pass, chunks
        this rank processed).  `on_encoded(first_image, enc)` gets the job-wide index of the chunk's first
        image."""
        assert job.in_shape[1:] == (self.h, self.w, 3) and job.n % self.chunk == 0
        per_rank = job.n // self.chunk
        total = repeat * job.world * per_rank
        done = [0] * self.slots

        def tickets(slot):
            while True:
                v = job.take()
                if v >= total:
                    return
                done[slot] += 1
                u = v % (job.world * per_rank)
                owner, c = u // per_rank, u % per_rank
                a, b = c * self.chunk, (c + 1) * self.chunk
                yield v, owner * job.n + a, job.inputs[owner][a:b], job.outputs[owner][a:b], v < job.world * per_rank

        payload, _ = self._run(tickets, on_encoded, trace, False, from_device, copy_only)
        return payload, sum(done)

    def _run(self, tickets, on_encoded, trace, resident, from_device, copy_only):
        import threading
        import time
        totals = [0] * self.slots
        errors = []
        gate_in, gate_out = threading.Lock(), threading.Lock()

        def work(slot):
            try:
                if self.device is not None:
                    _lib.check(_lib.load().hic_set_device(int(self.device)))
                codec = self.codecs[slot]
                for v, first_image, src, dst, count_payload in tickets(slot):
                    t0 = time.perf_counter()
                    with gate_in:
                        t1 = time.perf_counter()
                        if not resident:
                            codec.upload(src)
                            _lib.sync(codec.stream)
                    t2 = time.perf_counter()
                    if copy_only:
                        codec.download_payload_sized()
                        t3 = t4 = time.perf_counter()
                    else:
                        enc = codec.encode_resident()
                        t3 = time.perf_counter()
                        if count_payload:
                            totals[slot] += int(enc.data.nbytes)
                        if on_encoded is not None:
                            on_encoded(first_image, enc)
                        if from_device:
                            codec.decode_device()
                        else:
                            codec.decode_resident(enc)
                        t4 = time.perf_counter()
                    with gate_out:
                        t5 = time.perf_counter()
                        if not resident:
                            codec.fetch(dst)
                        else:
                            _lib.sync(codec.stream)
                    t6 = time.perf_counter()
                    if trace is not None:
                        trace.append((slot, v, t0, t1, t2, t3, t4, t5, t6))
            except Exception as e:      # surfaced to the caller below
                errors.append(e)

        threads = [threading.Thread(target=work, args=(s,)) for s in range(self.slots)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errors:
            raise errors[0]
        return sum(totals), None

    def close(self):
        for c in self.codecs:
            c.close()
        for st in self.streams:
            _lib.stream_destroy(st)
        self.codecs, self.streams = [], []
