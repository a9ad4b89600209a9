"""Entropy stage plumbing shared by codec.py (single image, reference signatures) and batch.py.

Wraps the plan objects of include/hiccup_b200.h.  A symbol stream is indexed
s = (image * 3 + channel) * 3 + kind with kind 0 = DC differences, 1 = run-length values,
2 = run-length zero counts (channel order lum, cr, cb as in reference codec.py:304-317).
"""
import ctypes

import numpy as np

from hiccup_b200 import _lib

KIND_DC, KIND_VALUE, KIND_LENGTH = 0, 1, 2
DEFAULT_VALUE_BINS = 8192


CODE_MASK = np.uint64((1 << 58) - 1)


class EncodedStreams:
    """Host-side result of the entropy encoder for a batch: code tables and framed bit payloads.

    Tables are kept in the packed layout of hic_entropy_tables_packed: `index[s] = (first row, rows)`
    of symbol stream s, `symbols[r]`, `packed[r] = length << 58 | code bits`; a stream's rows are
    contiguous and in first-occurrence order."""

    def __init__(self, layout, index, nsym, nbits, byte_off, byte_len, symbols, packed, data):
        self.layout = layout
        self.index = np.asarray(index, np.uint32).reshape(-1, 2)
        self.nsym, self.nbits = nsym, nbits
        self.byte_off, self.byte_len = byte_off, byte_len
        self.symbols, self.packed = symbols, packed
        self.data = data                                   # uint8, all framed payloads, 4-byte aligned each

    @classmethod
    def from_tables(cls, layout, rows, nsym, nbits, byte_off, byte_len, symbols, lens, codes, data):
        """From per-stream row counts and concatenated (symbol, length, code) arrays in stream order."""
        rows = np.asarray(rows, np.uint32)
        start = np.concatenate(([0], np.cumsum(rows, dtype=np.uint64)[:-1])).astype(np.uint32)
        packed = (np.asarray(lens, np.uint64) << np.uint64(58)) | (np.asarray(codes, np.uint64) & CODE_MASK)
        return cls(layout, np.stack([start, rows], axis=1), nsym, nbits, byte_off, byte_len,
                   np.asarray(symbols, np.int32), packed, data)

    @property
    def rows(self):
        return self.index[:, 1]

    @property
    def total_rows(self):
        return int(self.index[:, 1].sum(dtype=np.uint64))

    def stream_rows(self, s):
        """(symbols, lengths, codes) of symbol stream s in first-occurrence order."""
        a = int(self.index[s, 0])
        b = a + int(self.index[s, 1])
        pk = self.packed[a:b]
        return self.symbols[a:b], (pk >> np.uint64(58)).astype(np.uint8), pk & CODE_MASK

    def table(self, s):
        """[(symbol, code string)] of symbol stream s in first-occurrence order."""
        sym, lens, codes = self.stream_rows(s)
        return [(int(v), format(int(code), "0%db" % int(ln))) for v, ln, code in zip(sym, lens, codes)]

    def framed(self, s):
        """The framed bytes of symbol stream s (what iohelper.padded_bs_2_bytes returns)."""
        a = int(self.byte_off[s])
        return self.data[a:a + int(self.byte_len[s])].tobytes()


class EntropyEncoder:
    """Owns a device plan for one batch shape; reusable across batches."""

    def __init__(self, layout, value_bins=DEFAULT_VALUE_BINS):
        _lib.require_device()
        self.lib = _lib.load()
        self.layout = layout
        self.value_bins = value_bins
        self.n_streams = layout.n_images * 9
        p = ctypes.c_void_p()
        _lib.check(self.lib.hic_entropy_plan_create(ctypes.byref(layout), value_bins, ctypes.byref(p)))
        self.plan = p
        self._out = None

    def close(self):
        if self.plan:
            self.lib.hic_entropy_plan_destroy(self.plan)
            self.plan = None
        if self._out is not None:
            self._out.free()
            self._out = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def symbolize(self, d_coef, stream=None):
        _lib.check(self.lib.hic_entropy_symbolize(self.plan, d_coef, stream))

    # ---- row-band sharding: two-pass E1 with the seam state in between, external codes ----------
    def scan(self, d_coef, stream=None):
        """Pass 1.  Returns (first_nz, last_nz) int32 arrays over the channel streams (-1: none)."""
        n_cs = self.layout.n_images * 3
        first, last = np.empty(n_cs, np.int32), np.empty(n_cs, np.int32)
        _lib.check(self.lib.hic_entropy_scan(self.plan, d_coef, first.ctypes.data, last.ctypes.data, stream))
        return first, last

    def emit(self, d_coef, band=None, stream=None):
        """Pass 2.  band: list of (carry_zeros, prev_dc, more_after, closes_stream) per channel stream."""
        arr = None
        if band is not None:
            arr = (_lib.BandCarry * len(band))(*[_lib.BandCarry(*[int(v) for v in b]) for b in band])
        _lib.check(self.lib.hic_entropy_emit(self.plan, d_coef, arr, stream))

    def histograms(self, stream=None):
        """Compacted histograms of the last emit: (index (n_streams, 2), entries (n, 3) int32 rows of
        (symbol, count, first occurrence), run-length symbol count per channel stream)."""
        index = np.empty(2 * self.n_streams, np.uint32)
        nsym_rl = np.empty(self.layout.n_images * 3, np.uint32)
        n = ctypes.c_uint64(0)
        _lib.check(self.lib.hic_entropy_histograms(self.plan, index.ctypes.data, None, 0, ctypes.byref(n), nsym_rl.ctypes.data, stream))
        entries = np.empty((max(int(n.value), 1), 3), np.int32)
        _lib.check(self.lib.hic_entropy_histograms(self.plan, index.ctypes.data, entries.ctypes.data, entries.shape[0],
                                                   ctypes.byref(n), nsym_rl.ctypes.data, stream))
        return index.reshape(-1, 2), entries[:int(n.value)], nsym_rl

    def set_codes(self, index, symbols, packed, nsym, nbits, start_bit=None, stream=None):
        """Install externally built codes (packed table layout) and this plan's symbol / bit counts."""
        index = np.ascontiguousarray(index, np.uint32)
        symbols = np.ascontiguousarray(symbols, np.int32)
        packed = np.ascontiguousarray(packed, np.uint64)
        nsym = np.ascontiguousarray(nsym, np.uint32)
        nbits = np.ascontiguousarray(nbits, np.uint64)
        sb = None if start_bit is None else np.ascontiguousarray(start_bit, np.uint32)
        _lib.check(self.lib.hic_entropy_set_codes(self.plan, index.ctypes.data, symbols.ctypes.data, packed.ctypes.data,
                                                  int(symbols.size), nsym.ctypes.data, nbits.ctypes.data,
                                                  None if sb is None else sb.ctypes.data, stream))
        n = self.n_streams
        self.rows, self.nsym = np.zeros(n, np.uint32), np.zeros(n, np.uint32)
        self.nbits, self.byte_off, self.byte_len = np.zeros(n, np.uint64), np.zeros(n, np.uint64), np.zeros(n, np.uint64)
        tr, tb = ctypes.c_uint64(0), ctypes.c_uint64(0)
        _lib.check(self.lib.hic_entropy_stream_info(self.plan, self.rows.ctypes.data, self.nsym.ctypes.data,
                                                    self.nbits.ctypes.data, self.byte_off.ctypes.data,
                                                    self.byte_len.ctypes.data, ctypes.byref(tr), ctypes.byref(tb)))
        self.total_rows, self.total_bytes = tr.value, tb.value

    def build_codes(self, stream=None, on_device=False):
        """E2.  on_device=False: host heapq replay (reference-faithful default, any alphabet size);
        on_device=True: the same replay by one CTA per stream on the GPU (alphabets <= 8192)."""
        if on_device:
            _lib.check(self.lib.hic_entropy_build_codes_device(self.plan, stream))
        else:
            _lib.check(self.lib.hic_entropy_build_codes(self.plan, stream))
        n = self.n_streams
        self.rows = np.zeros(n, np.uint32)
        self.nsym = np.zeros(n, np.uint32)
        self.nbits = np.zeros(n, np.uint64)
        self.byte_off = np.zeros(n, np.uint64)
        self.byte_len = np.zeros(n, np.uint64)
        tr, tb = ctypes.c_uint64(0), ctypes.c_uint64(0)
        _lib.check(self.lib.hic_entropy_stream_info(self.plan, self.rows.ctypes.data, self.nsym.ctypes.data,
                                                    self.nbits.ctypes.data, self.byte_off.ctypes.data,
                                                    self.byte_len.ctypes.data, ctypes.byref(tr), ctypes.byref(tb)))
        self.total_rows, self.total_bytes = tr.value, tb.value

    def tables(self):
        sym = np.zeros(self.total_rows, np.int32)
        lens = np.zeros(self.total_rows, np.uint8)
        codes = np.zeros(self.total_rows, np.uint64)
        _lib.check(self.lib.hic_entropy_tables(self.plan, sym.ctypes.data, lens.ctypes.data, codes.ctypes.data))
        return sym, lens, codes

    def tables_packed(self, stream=None, out=None):
        """(index, symbols, packed) as EncodedStreams wants them.  `out`: preallocated (pinned) arrays
        (index uint32[2 n_streams], symbols int32[>= total_rows], packed uint64[>= total_rows]).
        Synchronises `stream`."""
        n = int(self.total_rows)
        if out is None:
            out = (np.empty(2 * self.n_streams, np.uint32), np.empty(max(n, 1), np.int32), np.empty(max(n, 1), np.uint64))
        index, sym, packed = out
        assert index.size >= 2 * self.n_streams and sym.size >= n and packed.size >= n
        _lib.check(self.lib.hic_entropy_tables_packed(self.plan, index.ctypes.data, sym.ctypes.data, packed.ctypes.data, stream))
        _lib.sync(stream)
        return index[:2 * self.n_streams].reshape(-1, 2), sym[:n], packed[:n]

    def pack(self, stream=None):
        """Returns the device buffer holding all framed payloads (valid until the next pack)."""
        need = int(self.total_bytes) + 16
        if self._out is None or self._out.nbytes < need:
            if self._out is not None:
                self._out.free()
            self._out = _lib.DeviceBuffer(need + need // 4)
        _lib.check(self.lib.hic_entropy_pack(self.plan, self._out.ptr, stream))
        return self._out

    def device_tables(self):
        """Device pointers (index, row symbols, packed rows) for EntropyDecoder.set_tables_device."""
        ptrs = [ctypes.c_void_p() for _ in range(5)]
        _lib.check(self.lib.hic_entropy_device_tables(self.plan, *[ctypes.byref(q) for q in ptrs]))
        return tuple(q.value for q in ptrs)

    def encode(self, d_coef, stream=None, download=True, on_device=False):
        """Full entropy encode of device-resident zigzag blocks."""
        self.symbolize(d_coef, stream)
        self.build_codes(stream, on_device=on_device)
        out = self.pack(stream)
        if not download:
            _lib.sync(stream)
            return None
        data = out.download(np.uint8, int(self.total_bytes), stream)
        index, sym, packed = self.tables_packed(stream)
        return EncodedStreams(self.layout, index, self.nsym, self.nbits, self.byte_off, self.byte_len, sym, packed, data)

    def symbol_arrays(self, stream=None):
        """Download DC differences and run-length symbols (tests / band stitching)."""
        d_dc, d_val, d_len = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_void_p()
        _lib.check(self.lib.hic_entropy_symbol_buffers(self.plan, ctypes.byref(d_dc), ctypes.byref(d_val),
                                                       ctypes.byref(d_len)))
        lay = self.layout
        total_blocks = lay.n_images * lay.blocks_per_image
        dc = np.empty(total_blocks, np.int16)
        val = np.empty(total_blocks * 64, np.int16)
        ln = np.empty(total_blocks * 64, np.uint8)
        _lib.check(self.lib.hic_memcpy_d2h(dc.ctypes.data, d_dc, dc.nbytes, stream))
        _lib.check(self.lib.hic_memcpy_d2h(val.ctypes.data, d_val, val.nbytes, stream))
        _lib.check(self.lib.hic_memcpy_d2h(ln.ctypes.data, d_len, ln.nbytes, stream))
        _lib.sync(stream)
        return dc, val, ln


class EntropyDecoder:
    def __init__(self, layout):
        _lib.require_device()
        self.lib = _lib.load()
        self.layout = layout
        self.n_streams = layout.n_images * 9
        p = ctypes.c_void_p()
        _lib.check(self.lib.hic_decode_plan_create(ctypes.byref(layout), ctypes.byref(p)))
        self.plan = p
        self._in = None

    def close(self):
        if self.plan:
            self.lib.hic_decode_plan_destroy(self.plan)
            self.plan = None
        if self._in is not None:
            self._in.free()
            self._in = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_tables_device(self, d_index, d_row_sym, d_row_packed, total_rows, stream=None):
        _lib.check(self.lib.hic_decode_set_tables_device(self.plan, d_index, d_row_sym, d_row_packed, int(total_rows), stream))

    def run(self, d_data, byte_off, nbits, d_coef, stream=None):
        byte_off = np.ascontiguousarray(byte_off, np.uint64)
        nbits = np.ascontiguousarray(nbits, np.uint64)
        _lib.check(self.lib.hic_decode_run(self.plan, d_data, byte_off.ctypes.data, nbits.ctypes.data, d_coef, stream))

    def decode_device_data(self, index, symbols, packed, d_data, byte_off, nbits, d_coef, stream=None):
        """Packed host tables + framed payloads already on the device (d_data: pointer; byte_off 4-byte aligned)."""
        index = np.ascontiguousarray(index, np.uint32)
        symbols = np.ascontiguousarray(symbols, np.int32)
        packed = np.ascontiguousarray(packed, np.uint64)
        _lib.check(self.lib.hic_decode_set_tables_packed(self.plan, index.ctypes.data, symbols.ctypes.data,
                                                         packed.ctypes.data, int(symbols.size), stream))
        self.run(d_data, byte_off, nbits, d_coef, stream)                     # synchronises: host arrays may go

    def decode_streams(self, enc, d_coef, stream=None):
        """Decode an EncodedStreams (packed tables; no per-row host work)."""
        index = np.ascontiguousarray(enc.index, np.uint32)
        symbols = np.ascontiguousarray(enc.symbols, np.int32)
        packed = np.ascontiguousarray(enc.packed, np.uint64)
        total = int(symbols.size)
        _lib.check(self.lib.hic_decode_set_tables_packed(self.plan, index.ctypes.data, symbols.ctypes.data,
                                                         packed.ctypes.data, total, stream))
        data = np.ascontiguousarray(enc.data, np.uint8)
        need = data.nbytes + 16
        if self._in is None or self._in.nbytes < need:
            if self._in is not None:
                self._in.free()
            self._in = _lib.DeviceBuffer(need + need // 4)
        self._in.upload(data, stream)
        self.run(self._in.ptr, enc.byte_off, enc.nbits, d_coef, stream)      # synchronises: host arrays may go

    @staticmethod
    def subsequences(nbits):
        """128-bit subsequences of each stream (one restart record each): the 8 framing bits count."""
        return [(8 + int(b) + 127) // 128 if int(b) else 0 for b in nbits]

    def decode(self, rows, symbols, lens, codes, data, byte_off, nbits, d_coef, stream=None, d_data=None, restarts=None,
               sync_only=False):
        """rows/symbols/lens/codes: concatenated code tables; data: uint8 host array holding every
        framed payload at byte_off[s] (4-byte aligned); nbits[s]: payload bits.  Fills d_coef.
        restarts = (off, cnt): the restart records of every subsequence in stream order (the `.hic` extension):
        the synchronisation passes are skipped.  sync_only: run only those passes and return the records."""
        rows = np.ascontiguousarray(rows, np.uint32)
        symbols = np.ascontiguousarray(symbols, np.int32)
        lens = np.ascontiguousarray(lens, np.uint8)
        codes = np.ascontiguousarray(codes, np.uint64)
        byte_off = np.ascontiguousarray(byte_off, np.uint64)
        nbits = np.ascontiguousarray(nbits, np.uint64)
        _lib.check(self.lib.hic_decode_set_tables(self.plan, rows.ctypes.data, symbols.ctypes.data, lens.ctypes.data,
                                                  codes.ctypes.data, stream))
        if d_data is None:
            data = np.ascontiguousarray(data, np.uint8)
            need = data.nbytes + 16
            if self._in is None or self._in.nbytes < need:
                if self._in is not None:
                    self._in.free()
                self._in = _lib.DeviceBuffer(need + need // 4)
            self._in.upload(data, stream)
            d_data = self._in.ptr
            _lib.check(self.lib.hic_decode_set_data_bytes(self.plan, int(data.nbytes)))
        else:
            _lib.check(self.lib.hic_decode_set_data_bytes(self.plan, 0))
        if sync_only:
            n_sub = ctypes.c_uint64()
            _lib.check(self.lib.hic_decode_sync(self.plan, d_data, byte_off.ctypes.data, nbits.ctypes.data, ctypes.byref(n_sub), stream))
            off, cnt = np.empty(n_sub.value, np.uint8), np.empty(n_sub.value, np.uint8)
            _lib.check(self.lib.hic_decode_export_restarts(self.plan, off.ctypes.data, cnt.ctypes.data, n_sub.value, stream))
            return off, cnt
        if restarts is not None:
            off = np.ascontiguousarray(restarts[0], np.uint8)
            cnt = np.ascontiguousarray(restarts[1], np.uint8)
            assert off.size == cnt.size
            _lib.check(self.lib.hic_decode_run_restarts(self.plan, d_data, byte_off.ctypes.data, nbits.ctypes.data,
                                                        off.ctypes.data, cnt.ctypes.data, int(off.size), d_coef, stream))
            return None
        _lib.check(self.lib.hic_decode_run(self.plan, d_data, byte_off.ctypes.data, nbits.ctypes.data, d_coef, stream))
        return None

    def run_dc(self, d_data, byte_off, nbits, d_dc, stream=None, restarts=None):
        """DC-only decode (hic_decode_run_dc) with the tables already installed: d_dc receives one int16 DC value per
        block.  Only the DC streams' entries of byte_off / nbits and their bytes are read.  restarts = (off, cnt): the
        DC streams' records in stream order; records that do not fit mean decoding the long way (and failing there
        if the streams are bad), never a silent mis-decode."""
        byte_off = np.ascontiguousarray(byte_off, np.uint64)
        nbits = np.ascontiguousarray(nbits, np.uint64)
        if restarts is not None:
            off = np.ascontiguousarray(restarts[0], np.uint8)
            cnt = np.ascontiguousarray(restarts[1], np.uint8)
            assert off.size == cnt.size
            try:
                _lib.check(self.lib.hic_decode_run_dc(self.plan, d_data, byte_off.ctypes.data, nbits.ctypes.data,
                                                      off.ctypes.data, cnt.ctypes.data, int(off.size), d_dc, stream))
                return True
            except _lib.HicError:
                pass
        _lib.check(self.lib.hic_decode_run_dc(self.plan, d_data, byte_off.ctypes.data, nbits.ctypes.data, None, None, 0, d_dc, stream))
        return False

    def decode_dc(self, index, symbols, packed, data, byte_off, nbits, d_dc, stream=None, restarts=None):
        """Packed host tables (the AC streams may have no rows) + framed payloads in a host array (the DC streams'
        bytes at least) -> run_dc.  The data bound is checked against `data`.  Returns whether the records were used."""
        index = np.ascontiguousarray(index, np.uint32)
        symbols = np.ascontiguousarray(symbols, np.int32)
        packed = np.ascontiguousarray(packed, np.uint64)
        _lib.check(self.lib.hic_decode_set_tables_packed(self.plan, index.ctypes.data, symbols.ctypes.data,
                                                         packed.ctypes.data, int(symbols.size), stream))
        data = np.ascontiguousarray(data, np.uint8)
        need = data.nbytes + 16
        if self._in is None or self._in.nbytes < need:
            if self._in is not None:
                self._in.free()
            self._in = _lib.DeviceBuffer(need + need // 4)
        self._in.upload(data, stream)
        _lib.check(self.lib.hic_decode_set_data_bytes(self.plan, int(data.nbytes)))
        try:
            return self.run_dc(self._in.ptr, byte_off, nbits, d_dc, stream, restarts)
        finally:
            _lib.check(self.lib.hic_decode_set_data_bytes(self.plan, 0))


def dc_streams_only(enc):
    """The DC streams of an EncodedStreams alone, for decode_dc: (index, symbols, packed, data, byte_off, nbits) with
    the AC streams at zero rows and zero bits, and the DC streams' tables and framed bytes packed together."""
    n_s = enc.index.shape[0]
    dc = np.arange(0, n_s, 3)
    start = enc.index[dc, 0].astype(np.int64)
    rows = enc.index[dc, 1].astype(np.int64)
    index = np.zeros((n_s, 2), np.uint32)
    index[dc, 1] = rows
    index[dc, 0] = np.concatenate(([0], np.cumsum(rows)[:-1])).astype(np.uint32)
    b_off = np.asarray(enc.byte_off, np.int64)[dc]
    b_len = np.asarray(enc.byte_len, np.int64)[dc]
    b_pad = (b_len + 3) & ~3                                             # whole words: every stream starts 4-byte aligned
    byte_off = np.zeros(n_s, np.uint64)
    byte_off[dc] = np.concatenate(([0], np.cumsum(b_pad)[:-1])).astype(np.uint64)
    data = np.zeros(int(b_pad.sum()) + 16, np.uint8)
    src = np.asarray(enc.data, np.uint8)
    # slices, one per stream: a few thousand of them cost less than an element-wise gather of megabytes
    for a, o, n in zip(byte_off[dc].tolist(), b_off.tolist(), b_len.tolist()):
        data[a:a + n] = src[o:o + n]
    symbols, packed = np.asarray(enc.symbols), np.asarray(enc.packed)
    pick = [slice(a, a + n) for a, n in zip(start.tolist(), rows.tolist())]
    cat = lambda arr: np.concatenate([arr[s] for s in pick]) if pick else arr[:0]
    nbits = np.zeros(n_s, np.uint64)
    nbits[dc] = np.asarray(enc.nbits, np.uint64)[dc]
    return index, cat(symbols), cat(packed), data, byte_off, nbits


# ------------------------------------------------------------------------------------------------
# plan cache of the single-image entry points (codec.jpeg_encode / jpeg_decode / wavelet_*): an entropy plan
# is some forty device allocations, and an image-at-a-time caller (run.compress over a directory, the
# reference's own usage) keeps asking for the same shape.  A few plans per thread, least recently used out.
# ------------------------------------------------------------------------------------------------
import threading

_PLAN_CACHE = threading.local()
PLAN_CACHE_SIZE = 4


def _layout_key(layout):
    return (int(layout.n_images), int(layout.skip_first), int(layout.blocks_per_image), tuple(int(v) for v in layout.nb),
            tuple(int(v) for v in layout.block_off), tuple(int(v) for v in layout.len))


def _cached(kind, key, make):
    cache = getattr(_PLAN_CACHE, "plans", None)
    if cache is None:
        cache = _PLAN_CACHE.plans = []            # [(kind, key, object)], most recent last
    for i, (k, q, obj) in enumerate(cache):
        if k == kind and q == key:
            cache.append(cache.pop(i))
            return obj
    obj = make()
    cache.append((kind, key, obj))
    while len(cache) > PLAN_CACHE_SIZE:
        cache.pop(0)[2].close()
    return obj


def cached_encoder(layout, value_bins=DEFAULT_VALUE_BINS):
    """An EntropyEncoder for this layout that outlives the call (do not close it)."""
    key = (_lib.current_device(), _layout_key(layout), int(value_bins))
    return _cached("enc", key, lambda: EntropyEncoder(layout, value_bins))


def cached_decoder(layout):
    """An EntropyDecoder for this layout that outlives the call (do not close it)."""
    key = (_lib.current_device(), _layout_key(layout))
    return _cached("dec", key, lambda: EntropyDecoder(layout))


def drop_cached_plans():
    cache = getattr(_PLAN_CACHE, "plans", None) or []
    while cache:
        cache.pop()[2].close()
