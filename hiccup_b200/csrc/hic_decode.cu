// hic_decode.cu -- entropy decode stage: Huffman decode (D1), run-length expansion (D2), DC prefix
// sum and de-zigzag into blocks (D3).
//
// The `.hic` format carries no restart offsets (codec.py:319-334); D1 recovers parallelism inside a
// stream from the self-synchronising property of Huffman codes.  D2 and D3 are tile scans over the
// decoded symbols.
#include <algorithm>
#include <vector>
#include "hic_core.cuh"
#include "hic_runtime.cuh"

namespace hic {
namespace dec {

constexpr int XT = 2048;             // symbols per expand tile
constexpr int XTHREADS = 256;
constexpr int XSPT = XT / XTHREADS;

struct RowIndex {       // rows of one symbol stream inside the row arrays (same layout as the encoder's index)
    uint32_t offset, count;
};

struct Geom {
    hic_stream_layout L;
    int xtiles[3];              // expand tiles per channel (capacity = 64 * nb symbols)
    int xtiles_per_image;
    int dtiles[3];              // DC tiles per channel (capacity = nb)
    int dtiles_per_image;
};

__host__ __device__ inline int64_t cs_block_base(const Geom& g, int img, int c) {
    return (int64_t)img * g.L.blocks_per_image + g.L.block_off[c];
}

// ------------------------------------------------------------------------------------------------
// D1: parallel Huffman decode by self-synchronisation.
//
// The format has no restart offsets, but Huffman codes self-synchronise: a decoder started at an
// arbitrary bit falls onto true codeword boundaries after a few symbols.  Each stream is cut into
// subsequences of SUB_BITS bits, one thread each; a CTA owns SUB_PER_CTA consecutive subsequences.
//   sync kernel   every thread decodes from its nominal start until it crosses its upper boundary
//                 and records where it stopped; then, in a loop inside the CTA, thread t restarts
//                 from where thread t-1 stopped until nothing changes (shared memory only);
//   resync kernel the same, seeded with the stop position of the previous CTA's last thread;
//                 relaunched until no CTA's last stop position changes (usually once);
//   count scan    symbols per CTA -> output offsets (per-stream scan);
//   write kernel  final pass from the now-correct starts, writing symbols at their offsets.
// Code lookup: a 12-bit first-level table in shared memory; prefixes of longer codes point into a
// per-stream second-level table of up to 8 more bits; a code that runs past 20 bits (or a prefix
// the second level had no room for) is found by predecessor search over the stream's rows sorted by
// left-aligned code -- prefix-free codes are disjoint intervals of the 64-bit window space.
// ------------------------------------------------------------------------------------------------
constexpr int L1_BITS = 12;
constexpr int L1_SIZE = 1 << L1_BITS;
constexpr int L2_MAX_EXTRA = 8;
constexpr int L2_CAP_MIN = 4096;             // second-level entries per stream: the plan picks a power of two
constexpr int L2_CAP_MAX = 65536;            // in this range from a budget of 2^28 entries per plan
constexpr int L2_LONG = 0xFF;                // second-level length field: the code runs past 20 bits
constexpr int SUB_BITS = 128;
constexpr int SUB_PER_CTA = 256;
constexpr int CHUNK_WORDS = SUB_BITS * SUB_PER_CTA / 32;      // 1024 words of bit stream per CTA
constexpr int CHUNK_SLACK = 8;                                // a code may run 58 bits past the last boundary
constexpr int L1_FALLBACK = 0xFF;
constexpr int PK_BITS = 10;                  // window of the packed multi-symbol table of the zero-count streams
constexpr int PK_SIZE = 1 << PK_BITS;
constexpr int PK_MAX_SYMS = 5;

struct SyncTile {
    uint32_t ss;            // symbol stream
    uint32_t sub0;          // first subsequence of the tile inside its stream
    uint64_t sub_base;      // global index of that subsequence
};

// one CTA per symbol stream: first- and second-level tables from the code rows; streams that own a
// code longer than 20 bits (or overflow the second level) also get their rows sorted by
// left-aligned code for the predecessor search.
__global__ void __launch_bounds__(256)
build_tables_kernel(const RowIndex* __restrict__ index, const int32_t* __restrict__ row_sym,
                    const uint64_t* __restrict__ row_packed, int32_t* __restrict__ lut1, int32_t* __restrict__ lut2,
                    int l2_cap, uint64_t* __restrict__ sorted_left, uint32_t* __restrict__ sorted_row,
                    uint16_t* __restrict__ mlut, uint32_t* __restrict__ pklut) {
    __shared__ uint32_t extra[L1_SIZE];          // max (len - 12) under each 12-bit prefix
    __shared__ uint32_t offs[L1_SIZE];
    __shared__ uint32_t wsum[8];
    __shared__ int s_need_sort;
    const int ss = blockIdx.x;
    int32_t* my1 = lut1 + (size_t)ss * L1_SIZE;
    int32_t* my2 = lut2 + (size_t)ss * l2_cap;
    for (int i = threadIdx.x; i < L1_SIZE; i += blockDim.x) {
        my1[i] = 0;
        extra[i] = 0;
    }
    if (threadIdx.x == 0) s_need_sort = 0;
    __syncthreads();
    const uint64_t r0 = index[ss].offset, r1 = r0 + index[ss].count;
    constexpr uint64_t CODE_MASK = (1ull << 58) - 1;
    // A code of `len` <= 12 bits owns 2^(12 - len) consecutive first-level entries: a warp takes 32 rows at a
    // time and all its lanes fill each row's span together (one thread alone would write 2048 entries for a
    // 1-bit code while the rest of the CTA waits).
    for (uint64_t rb = r0 + (threadIdx.x & ~31u); rb < r1; rb += blockDim.x) {
        const uint64_t r = rb + (threadIdx.x & 31);
        uint32_t span = 0, base = 0;
        int32_t entry = 0;
        if (r < r1) {
            const uint32_t len = (uint32_t)(row_packed[r] >> 58);
            const uint64_t code = row_packed[r] & CODE_MASK;
            if (len != 0 && len <= L1_BITS) {
                base = (uint32_t)(code << (L1_BITS - len));
                entry = (row_sym[r] << 8) | (int32_t)len;
                span = 1u << (L1_BITS - len);
            } else if (len != 0) {
                atomicMax(&extra[(uint32_t)(code >> (len - L1_BITS))], min(len - L1_BITS, (uint32_t)L2_MAX_EXTRA));
                if (len > L1_BITS + L2_MAX_EXTRA) s_need_sort = 1;
            }
        }
        unsigned todo = __ballot_sync(0xffffffffu, span != 0);
        while (todo) {
            const int k = __ffs(todo) - 1;
            todo &= todo - 1;
            const uint32_t n = __shfl_sync(0xffffffffu, span, k), b = __shfl_sync(0xffffffffu, base, k);
            const int32_t e = __shfl_sync(0xffffffffu, entry, k);
            for (uint32_t j = threadIdx.x & 31; j < n; j += 32) my1[b + j] = e;
        }
    }
    __syncthreads();
    // exclusive scan of the second-level sizes over the 4096 prefixes (16 per thread)
    uint32_t local[16], sum = 0;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const uint32_t e = extra[threadIdx.x * 16 + j];
        local[j] = e ? (1u << e) : 0u;
        sum += local[j];
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = sum;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const uint32_t o = __shfl_up_sync(0xffffffffu, inc, off);
        if (lane >= off) inc += o;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    uint32_t run = inc - sum;
    for (int w = 0; w < warp; ++w) run += wsum[w];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const int pfx = threadIdx.x * 16 + j;
        const uint32_t e = extra[pfx];
        if (e) {
            if (run + local[j] <= (uint32_t)l2_cap) {
                offs[pfx] = run;
                my1[pfx] = (int32_t)((run << 8) | 0x80u | e);
            } else {
                offs[pfx] = 0xFFFFFFFFu;          // no room: the whole prefix goes to the search
                my1[pfx] = L1_FALLBACK;
                s_need_sort = 1;
            }
            run += local[j];
        }
    }
    if (threadIdx.x == blockDim.x - 1) wsum[0] = min(run, (uint32_t)l2_cap);      // second-level entries in use
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < wsum[0]; i += blockDim.x) my2[i] = 0;       // (incomplete code sets leave holes)
    __syncthreads();
    for (uint64_t r = r0 + threadIdx.x; r < r1; r += blockDim.x) {
        const uint32_t len = (uint32_t)(row_packed[r] >> 58);
        const uint64_t code = row_packed[r] & CODE_MASK;
        if (len <= L1_BITS) continue;
        const uint32_t pfx = (uint32_t)(code >> (len - L1_BITS));
        if (offs[pfx] == 0xFFFFFFFFu) continue;
        const uint32_t e = extra[pfx], x = len - L1_BITS;
        if (x <= e) {
            const uint32_t sub = (uint32_t)(code & ((1ull << x) - 1));
            const uint32_t base = offs[pfx] + (sub << (e - x));
            const int32_t entry = (row_sym[r] << 8) | (int32_t)len;
            for (uint32_t j = 0; j < (1u << (e - x)); ++j) my2[base + j] = entry;
        } else {                                   // longer than the second level reaches: mark its slot
            const uint32_t sub = (uint32_t)((code >> (x - e)) & ((1ull << e) - 1));
            my2[offs[pfx] + sub] = L2_LONG;
        }
    }
    // Multi-symbol table for the passes that only need positions and counts (the sync kernels): for every
    // 12-bit window, the whole codes that lie inside it -- low byte = their bits, high byte = how many
    // (0: the first code is longer than the window or unassigned; those are decoded one at a time).
    {
        __syncthreads();                           // `extra` is dead: it now holds a copy of the first-level table
        for (int i = threadIdx.x; i < L1_SIZE; i += blockDim.x) extra[i] = (uint32_t)my1[i];
        __syncthreads();
        uint16_t* mym = mlut + (size_t)ss * L1_SIZE;
        for (uint32_t pfx = threadIdx.x; pfx < (uint32_t)L1_SIZE; pfx += blockDim.x) {
            uint32_t pos = 0, cnt = 0;
            while (true) {
                const int32_t e = (int32_t)extra[(pfx << pos) & (L1_SIZE - 1)];
                const uint32_t len = (uint32_t)(e & 0x7F);
                if ((e & 0x80) || len == 0 || pos + len > (uint32_t)L1_BITS) break;
                pos += len;
                ++cnt;
            }
            mym[pfx] = (uint16_t)((cnt << 8) | pos);
        }
    }
    // Zero-count streams (symbols 0..14, short codes): the final decode also takes several symbols per
    // lookup.  For every PK_BITS-bit window: bits 0-2 = whole codes inside it (at most PK_MAX_SYMS),
    // bits 3-6 = their bits, bits 8.. = the symbols, 4 bits each.  A stream that owns a symbol outside
    // 0..15 (a foreign file) gets an all-zero table and is decoded one symbol at a time.
    if (ss % 3 == HIC_KIND_LENGTH) {
        __shared__ int s_wide;
        if (threadIdx.x == 0) s_wide = 0;
        __syncthreads();
        for (uint64_t r = r0 + threadIdx.x; r < r1; r += blockDim.x)
            if ((uint32_t)row_sym[r] > 15u) s_wide = 1;
        __syncthreads();
        uint32_t* myp = pklut + ((size_t)(ss / 3) * 2 + 1) * PK_SIZE;
        for (uint32_t w = threadIdx.x; w < (uint32_t)PK_SIZE; w += blockDim.x) {
            uint32_t pos = 0, cnt = 0, syms = 0;
            while (!s_wide && cnt < (uint32_t)PK_MAX_SYMS) {
                const int32_t e = (int32_t)extra[(w << (L1_BITS - PK_BITS + pos)) & (L1_SIZE - 1)];
                const uint32_t len = (uint32_t)(e & 0x7F);
                if ((e & 0x80) || len == 0 || pos + len > (uint32_t)PK_BITS) break;
                syms |= (uint32_t)((e >> 8) & 15) << (4 * cnt);
                pos += len;
                ++cnt;
            }
            myp[w] = cnt ? (cnt | (pos << 3) | (syms << 8)) : 0u;
        }
    }
    // Run-length value streams: pairs.  bits 0-1 = whole codes inside the window (at most 2) whose symbols
    // fit 12 signed bits, bits 2-5 = their bits, bits 8-19 and 20-31 = the symbols.
    if (ss % 3 == HIC_KIND_VALUE) {
        uint32_t* myp = pklut + (size_t)(ss / 3) * 2 * PK_SIZE;
        for (uint32_t w = threadIdx.x; w < (uint32_t)PK_SIZE; w += blockDim.x) {
            uint32_t pos = 0, cnt = 0, syms = 0;
            while (cnt < 2u) {
                const int32_t e = (int32_t)extra[(w << (L1_BITS - PK_BITS + pos)) & (L1_SIZE - 1)];
                const uint32_t len = (uint32_t)(e & 0x7F);
                const int32_t sym = e >> 8;
                if ((e & 0x80) || len == 0 || pos + len > (uint32_t)PK_BITS || sym < -2048 || sym > 2047) break;
                syms |= ((uint32_t)sym & 0xFFFu) << (12 * cnt);
                pos += len;
                ++cnt;
            }
            myp[w] = cnt ? (cnt | (pos << 2) | (syms << 8)) : 0u;
        }
    }
    if (!s_need_sort) return;
    // rows sorted by left-aligned code (bitonic, in global memory: only big alphabets come here)
    const uint32_t n = index[ss].count;
    uint32_t P = 1;
    while (P < n) P <<= 1;
    uint64_t* key = sorted_left + 2 * r0;          // room for the padded power of two
    uint32_t* row = sorted_row + 2 * r0;
    for (uint32_t i = threadIdx.x; i < P; i += blockDim.x) {
        if (i < n) {
            const uint64_t pk = row_packed[r0 + i];
            const uint32_t len = (uint32_t)(pk >> 58);
            key[i] = len ? (pk & CODE_MASK) << (64 - len) : ~0ull;
            row[i] = i;
        } else {
            key[i] = ~0ull;
            row[i] = 0xFFFFFFFFu;
        }
    }
    __syncthreads();
    for (uint32_t k = 2; k <= P; k <<= 1)
        for (uint32_t j = k >> 1; j > 0; j >>= 1) {
            for (uint32_t i = threadIdx.x; i < P; i += blockDim.x) {
                const uint32_t l = i ^ j;
                if (l > i) {
                    const bool up = (i & k) == 0;
                    const uint64_t ka = key[i], kb = key[l];
                    const uint32_t ra = row[i], rb = row[l];
                    // ties only among the padding; order them by row to keep the sort deterministic
                    const bool gt = ka > kb || (ka == kb && ra > rb);
                    if (gt == up) {
                        key[i] = kb;
                        key[l] = ka;
                        row[i] = rb;
                        row[l] = ra;
                    }
                }
            }
            __syncthreads();
        }
}

struct BitReader {
    const uint32_t* words;      // shared-memory copy of the CTA's chunk (already in MSB-first order)
    __device__ __forceinline__ uint64_t window(uint32_t rel_bit) const {
        const uint32_t wi = rel_bit >> 5, sh = rel_bit & 31;
        const uint64_t hi = ((uint64_t)words[wi] << 32) | words[wi + 1];
        return sh ? (hi << sh) | (words[wi + 2] >> (32 - sh)) : hi;
    }
};

struct LongSearch {            // per-stream view for the predecessor search
    const uint64_t* left;      // rows' left-aligned codes, ascending
    const uint32_t* row;       // row index (inside the stream) of each sorted entry
    const int32_t* row_sym;
    const uint64_t* row_packed;
    uint32_t n_rows;
};

// the row whose code is a prefix of the window, by predecessor search (prefix-free codes are disjoint
// intervals [code << (64 - len), (code + 1) << (64 - len)) of the window space)
__device__ __noinline__ uint32_t decode_long(uint64_t w, const LongSearch& ls, int32_t& sym) {
    if (ls.n_rows == 0) return 0;
    uint32_t lo = 0, hi = ls.n_rows;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(ls.left + mid) <= w) lo = mid; else hi = mid;
    }
    const uint32_t r = __ldg(ls.row + lo);
    if (r >= ls.n_rows) return 0;
    const uint64_t packed = __ldg(ls.row_packed + r);
    const uint32_t len = (uint32_t)(packed >> 58);
    if (len == 0 || (w >> (64 - len)) != (packed & ((1ull << 58) - 1))) return 0;
    sym = __ldg(ls.row_sym + r);
    return len;
}

// decode one code at the 64-bit window; returns its length (0 = no valid code) and the symbol
__device__ __forceinline__ uint32_t decode_one(uint64_t w, const int32_t* __restrict__ l1, const int32_t* __restrict__ l2,
                                               const LongSearch& ls, int32_t& sym) {
    int32_t e = l1[(uint32_t)(w >> (64 - L1_BITS))];
    if (!(e & 0x80)) {
        sym = e >> 8;
        return (uint32_t)(e & 0x7F);
    }
    const uint32_t nb2 = (uint32_t)(e & 0x7F);
    if (nb2 != 0x7F) {
        const uint32_t idx = ((uint32_t)e >> 8) + (uint32_t)((w >> (64 - L1_BITS - nb2)) & ((1u << nb2) - 1));
        e = __ldg(l2 + idx);
        if ((e & 0xFF) != L2_LONG) {
            sym = e >> 8;
            return (uint32_t)(e & 0xFF);
        }
    }
    return decode_long(w, ls, sym);
}

// Decode from `pos` until the position reaches `limit` (the thread's upper boundary) or `end`.
// Positions are bits from the stream's first byte; `chunk0` is the bit position of smem word 0.
template <bool WRITE>
__device__ __forceinline__ uint32_t decode_span(const BitReader& br, uint32_t chunk0, uint32_t pos, uint32_t limit,
                                                uint32_t end, const int32_t* __restrict__ l1,
                                                const int32_t* __restrict__ l2, const LongSearch& ls, uint32_t& count, int16_t* __restrict__ out16,
                                                uint8_t* __restrict__ out8, uint32_t out_idx, bool& bad) {
    count = 0;
    const uint32_t stop = limit < end ? limit : end;
    if (pos >= stop) return pos;
    // a 64-bit bit buffer, MSB first, refilled a word at a time: at least 32 valid bits at every lookup,
    // enough for both table levels (<= 20 bits); only the rare long codes rebuild a full 64-bit window
    uint32_t wi = (pos - chunk0) >> 5;
    const uint32_t sh = (pos - chunk0) & 31;
    uint64_t buf = (((uint64_t)br.words[wi] << 32) | br.words[wi + 1]) << sh;
    int avail = 64 - (int)sh;
    wi += 2;
    while (pos < stop) {
        if (avail < 32) {
            buf |= (uint64_t)br.words[wi] << (32 - avail);
            avail += 32;
            ++wi;
        }
        int32_t e = l1[(uint32_t)(buf >> (64 - L1_BITS))];
        uint32_t len;
        int32_t sym;
        if (!(e & 0x80)) {
            sym = e >> 8;
            len = (uint32_t)(e & 0x7F);
        } else {
            len = 0;
            sym = 0;
            const uint32_t nb2 = (uint32_t)(e & 0x7F);
            if (nb2 != 0x7F) {
                const uint32_t idx = ((uint32_t)e >> 8) + (uint32_t)((buf >> (64 - L1_BITS - nb2)) & ((1u << nb2) - 1));
                e = __ldg(l2 + idx);
                if ((e & 0xFF) != L2_LONG) {
                    sym = e >> 8;
                    len = (uint32_t)(e & 0xFF);
                } else {
                    len = decode_long(br.window(pos - chunk0), ls, sym);
                }
            } else {
                len = decode_long(br.window(pos - chunk0), ls, sym);
            }
        }
        if (len == 0 || pos + len > end) {
            bad = true;
            return stop;          // not a codeword boundary (or a corrupt stream): give up on this span
        }
        if (WRITE) {
            if (out8) out8[out_idx + count] = (uint8_t)sym; else out16[out_idx + count] = (int16_t)sym;
        }
        ++count;
        pos += len;
        if (len >= 32) {          // a long code: rebuild the buffer at the new position
            wi = (pos - chunk0) >> 5;
            const uint32_t s2 = (pos - chunk0) & 31;
            buf = (((uint64_t)br.words[wi] << 32) | br.words[wi + 1]) << s2;
            avail = 64 - (int)s2;
            wi += 2;
        } else {
            buf <<= len;
            avail -= (int)len;
        }
    }
    return pos;
}

// The sync kernels only need where a span ends and how many symbols it holds: while a 12-bit window
// cannot cross the span's upper boundary, one lookup in the multi-symbol table steps over every whole
// code inside the window (2.4 on average on the C2 streams); the last bits before the boundary, and codes
// longer than the window, go one symbol at a time exactly as in decode_span.
__device__ __forceinline__ uint32_t decode_span_count(const BitReader& br, uint32_t chunk0, uint32_t pos, uint32_t limit,
                                                      uint32_t end, const int32_t* __restrict__ l1,
                                                      const uint16_t* __restrict__ m1, const int32_t* __restrict__ l2,
                                                      const LongSearch& ls, uint32_t& count, bool& bad) {
    count = 0;
    const uint32_t stop = limit < end ? limit : end;
    if (pos >= stop) return pos;
    uint32_t wi = (pos - chunk0) >> 5;
    const uint32_t sh = (pos - chunk0) & 31;
    uint64_t buf = (((uint64_t)br.words[wi] << 32) | br.words[wi + 1]) << sh;
    int avail = 64 - (int)sh;
    wi += 2;
    while (pos < stop) {
        if (avail < 32) {
            buf |= (uint64_t)br.words[wi] << (32 - avail);
            avail += 32;
            ++wi;
        }
        const uint32_t window = (uint32_t)(buf >> (64 - L1_BITS));
        if (pos + L1_BITS <= stop) {
            const uint32_t m = m1[window];
            if (m) {
                const uint32_t adv = m & 0xFFu;
                count += m >> 8;
                pos += adv;
                buf <<= adv;
                avail -= (int)adv;
                continue;
            }
        }
        int32_t e = l1[window];
        uint32_t len;
        int32_t sym;
        if (!(e & 0x80)) {
            len = (uint32_t)(e & 0x7F);
        } else {
            len = 0;
            sym = 0;
            const uint32_t nb2 = (uint32_t)(e & 0x7F);
            if (nb2 != 0x7F) {
                const uint32_t idx = ((uint32_t)e >> 8) + (uint32_t)((buf >> (64 - L1_BITS - nb2)) & ((1u << nb2) - 1));
                e = __ldg(l2 + idx);
                if ((e & 0xFF) != L2_LONG) len = (uint32_t)(e & 0xFF);
                else len = decode_long(br.window(pos - chunk0), ls, sym);
            } else {
                len = decode_long(br.window(pos - chunk0), ls, sym);
            }
        }
        if (len == 0 || pos + len > end) {
            bad = true;
            return stop;          // not a codeword boundary (or a corrupt stream): give up on this span
        }
        ++count;
        pos += len;
        if (len >= 32) {          // a long code: rebuild the buffer at the new position
            wi = (pos - chunk0) >> 5;
            const uint32_t s2 = (pos - chunk0) & 31;
            buf = (((uint64_t)br.words[wi] << 32) | br.words[wi + 1]) << s2;
            avail = 64 - (int)s2;
            wi += 2;
        } else {
            buf <<= len;
            avail -= (int)len;
        }
    }
    return pos;
}

// The final decode of a zero-count stream into the staging area: while a PK_BITS-bit window cannot cross
// the span's upper boundary, one lookup in the packed table yields up to PK_MAX_SYMS symbols; the last bits
// before the boundary (and anything the table does not hold) go one symbol at a time as in decode_span.
// (T = uint8_t: zero counts, five 4-bit symbols per entry; T = int16_t: run-length values, two 12-bit ones)
template <typename T>
__device__ __forceinline__ uint32_t decode_span_packed(const BitReader& br, uint32_t chunk0, uint32_t pos, uint32_t limit,
                                                       uint32_t end, const int32_t* __restrict__ l1,
                                                       const uint32_t* __restrict__ pk, const int32_t* __restrict__ l2,
                                                       const LongSearch& ls, uint32_t& count, T* __restrict__ stage,
                                                       uint32_t out_idx, bool& bad) {
    constexpr bool BYTES = sizeof(T) == 1;
    count = 0;
    const uint32_t stop = limit < end ? limit : end;
    if (pos >= stop) return pos;
    uint32_t wi = (pos - chunk0) >> 5;
    const uint32_t sh = (pos - chunk0) & 31;
    uint64_t buf = (((uint64_t)br.words[wi] << 32) | br.words[wi + 1]) << sh;
    int avail = 64 - (int)sh;
    wi += 2;
    T* out = stage + out_idx;
    while (pos < stop) {
        if (avail < 32) {
            buf |= (uint64_t)br.words[wi] << (32 - avail);
            avail += 32;
            ++wi;
        }
        if (pos + PK_BITS <= stop) {
            const uint32_t m = pk[(uint32_t)(buf >> (64 - PK_BITS))];
            const uint32_t n = BYTES ? (m & 7u) : (m & 3u);
            if (n) {
                const uint32_t adv = BYTES ? ((m >> 3) & 15u) : ((m >> 2) & 15u);
                T* o = out + count;
                if (BYTES) {
                    o[0] = (T)((m >> 8) & 15u);
                    if (n > 1) o[1] = (T)((m >> 12) & 15u);
                    if (n > 2) o[2] = (T)((m >> 16) & 15u);
                    if (n > 3) o[3] = (T)((m >> 20) & 15u);
                    if (n > 4) o[4] = (T)((m >> 24) & 15u);
                    static_assert(PK_MAX_SYMS == 5, "five symbol fields");
                } else {
                    o[0] = (T)((int32_t)(m << 12) >> 20);
                    if (n > 1) o[1] = (T)((int32_t)m >> 20);
                }
                count += n;
                pos += adv;
                buf <<= adv;
                avail -= (int)adv;
                continue;
            }
        }
        int32_t e = l1[(uint32_t)(buf >> (64 - L1_BITS))];
        uint32_t len;
        int32_t sym;
        if (!(e & 0x80)) {
            sym = e >> 8;
            len = (uint32_t)(e & 0x7F);
        } else {
            len = 0;
            sym = 0;
            const uint32_t nb2 = (uint32_t)(e & 0x7F);
            if (nb2 != 0x7F) {
                const uint32_t idx = ((uint32_t)e >> 8) + (uint32_t)((buf >> (64 - L1_BITS - nb2)) & ((1u << nb2) - 1));
                e = __ldg(l2 + idx);
                if ((e & 0xFF) != L2_LONG) {
                    sym = e >> 8;
                    len = (uint32_t)(e & 0xFF);
                } else {
                    len = decode_long(br.window(pos - chunk0), ls, sym);
                }
            } else {
                len = decode_long(br.window(pos - chunk0), ls, sym);
            }
        }
        if (len == 0 || pos + len > end) {
            bad = true;
            return stop;
        }
        out[count] = (T)sym;
        ++count;
        pos += len;
        if (len >= 32) {
            wi = (pos - chunk0) >> 5;
            const uint32_t s2 = (pos - chunk0) & 31;
            buf = (((uint64_t)br.words[wi] << 32) | br.words[wi + 1]) << s2;
            avail = 64 - (int)s2;
            wi += 2;
        } else {
            buf <<= len;
            avail -= (int)len;
        }
    }
    return pos;
}

struct SyncArgs {
    const uint8_t* bytes;
    const uint64_t* byte_off;
    const uint64_t* nbits;
    const int32_t* lut1;
    const int32_t* lut2;
    const uint16_t* mlut;
    const uint32_t* pklut;
    int l2_cap;
    const uint64_t* sorted_left;
    const uint32_t* sorted_row;
    const RowIndex* index;
    const int32_t* row_sym;
    const uint64_t* row_packed;
    const SyncTile* tiles;
    uint32_t* sub_end;          // per subsequence: where its decoder stopped
    uint16_t* sub_cnt;          // per subsequence: symbols decoded
    uint32_t* tile_start;       // per tile: the start its first thread used
    uint32_t* tile_cnt;         // per tile: symbols
    uint32_t* changed;          // set when a tile's last stop position moved
};

__device__ __forceinline__ void stage_chunk(const SyncArgs& a, const SyncTile& t, uint32_t* s_words, int32_t* s_l1) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(a.bytes + a.byte_off[t.ss]) + (size_t)t.sub0 * (SUB_BITS / 32);
    const uint64_t total_bits = 8 + a.nbits[t.ss];
    const uint32_t total_words = (uint32_t)((total_bits + 31) >> 5);
    const uint32_t w0 = t.sub0 * (SUB_BITS / 32);
    for (int i = threadIdx.x; i < CHUNK_WORDS + CHUNK_SLACK; i += blockDim.x)
        s_words[i] = (w0 + i < total_words) ? __byte_perm(__ldg(src + i), 0, 0x0123) : 0u;
    const int32_t* l1 = a.lut1 + (size_t)t.ss * L1_SIZE;
    for (int i = threadIdx.x; i < L1_SIZE; i += blockDim.x) s_l1[i] = __ldg(l1 + i);
}

template <bool RESYNC>
__global__ void __launch_bounds__(SUB_PER_CTA)
huffman_sync_kernel(SyncArgs a) {
    __shared__ uint32_t s_words[CHUNK_WORDS + CHUNK_SLACK];
    __shared__ int32_t s_l1[L1_SIZE];
    __shared__ uint16_t s_m1[L1_SIZE];
    __shared__ uint32_t s_end[SUB_PER_CTA];
    __shared__ uint32_t s_red[SUB_PER_CTA / 32];
    const SyncTile t = a.tiles[blockIdx.x];
    const uint32_t end = (uint32_t)(8 + a.nbits[t.ss]);
    const uint32_t n_sub = (end + SUB_BITS - 1) / SUB_BITS;
    const uint32_t sub = t.sub0 + threadIdx.x;
    const bool active = sub < n_sub;
    const uint64_t g = t.sub_base + threadIdx.x;
    const uint32_t chunk0 = t.sub0 * SUB_BITS;
    const uint32_t limit = (sub + 1) * SUB_BITS;
    const uint32_t tile_true_start = t.sub0 == 0 ? 8u : (RESYNC ? a.sub_end[t.sub_base - 1] : chunk0);
    if (RESYNC) {
        if (tile_true_start == a.tile_start[blockIdx.x]) return;      // nothing upstream moved
    }
    stage_chunk(a, t, s_words, s_l1);
    {
        const uint32_t* m1 = reinterpret_cast<const uint32_t*>(a.mlut + (size_t)t.ss * L1_SIZE);
        for (int i = threadIdx.x; i < L1_SIZE / 2; i += blockDim.x) reinterpret_cast<uint32_t*>(s_m1)[i] = __ldg(m1 + i);
    }
    const BitReader br{s_words};
    const int32_t* l2 = a.lut2 + (size_t)t.ss * a.l2_cap;
    const RowIndex ridx = a.index[t.ss];
    const LongSearch ls{a.sorted_left + 2 * (size_t)ridx.offset, a.sorted_row + 2 * (size_t)ridx.offset,
                        a.row_sym + ridx.offset, a.row_packed + ridx.offset, ridx.count};
    __syncthreads();

    uint32_t start, my_end = 0, cnt = 0, old_last_end = 0;
    bool bad = false;
    if (!RESYNC) {
        start = threadIdx.x == 0 ? tile_true_start : sub * SUB_BITS;
        if (active) my_end = decode_span_count(br, chunk0, start, limit, end, s_l1, s_m1, l2, ls, cnt, bad);
    } else {
        // previous state: my stop position and count; my start was my left neighbour's stop
        my_end = active ? a.sub_end[g] : 0;
        cnt = active ? a.sub_cnt[g] : 0;
        start = threadIdx.x == 0 ? a.tile_start[blockIdx.x] : (active ? a.sub_end[g - 1] : 0);
        if (threadIdx.x == blockDim.x - 1 || sub == n_sub - 1) old_last_end = my_end;
    }
    s_end[threadIdx.x] = my_end;
    // intra-CTA synchronisation: restart from the left neighbour's stop until nothing changes
    for (int iter = 0; iter <= SUB_PER_CTA; ++iter) {
        __syncthreads();
        const uint32_t want = threadIdx.x == 0 ? tile_true_start : s_end[threadIdx.x - 1];
        const bool redo = active && want != start;
        __syncthreads();
        bool moved = false;
        if (redo) {
            start = want;
            bad = false;
            const uint32_t e = decode_span_count(br, chunk0, start, limit, end, s_l1, s_m1, l2, ls, cnt, bad);
            moved = e != my_end;
            my_end = e;
            s_end[threadIdx.x] = e;
        }
        if (!__syncthreads_or(moved)) break;
    }
    if (active) {
        a.sub_end[g] = my_end;
        a.sub_cnt[g] = (uint16_t)cnt;
    }
    // tile totals
    uint32_t v = active ? cnt : 0;
#pragma unroll
    for (int off = 16; off; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t tot = 0;
        for (int w = 0; w < SUB_PER_CTA / 32; ++w) tot += s_red[w];
        a.tile_cnt[blockIdx.x] = tot;
        a.tile_start[blockIdx.x] = tile_true_start;
    }
    if (RESYNC && active && (threadIdx.x == blockDim.x - 1 || sub == n_sub - 1) && my_end != old_last_end)
        atomicOr(a.changed, 1u);
}

// per-stream exclusive scan of the tile symbol counts (tiles of a stream are consecutive)
__global__ void sync_tile_scan_kernel(int n_ss, const uint32_t* __restrict__ ss_tile0, const uint32_t* __restrict__ tile_cnt,
                                      uint32_t* __restrict__ tile_off, uint32_t* __restrict__ nsym_out) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_ss) return;
    uint32_t run = 0;
    for (uint32_t t = ss_tile0[s]; t < ss_tile0[s + 1]; ++t) {
        tile_off[t] = run;
        run += tile_cnt[t];
    }
    nsym_out[s] = run;
}

// Restart records (the `.hic` extension of hiccup_b200/hicimage.py; the reference's format has none,
// codec.py:319-334): for every SUB_BITS-bit subsequence of a stream, one byte `off` = how many bits past the
// subsequence's upper boundary the first codeword that starts at or after it begins (< 58), and one byte
// `cnt` = how many codewords start inside the span that ends there (<= SUB_BITS).  They are exactly what the
// sync passes converge to; a decoder that has them skips those passes.  The write kernel still checks every
// span against them, so a wrong record is reported as corruption, never decoded silently.
__global__ void __launch_bounds__(SUB_PER_CTA)
restart_export_kernel(const SyncTile* __restrict__ tiles, const uint64_t* __restrict__ nbits, const uint32_t* __restrict__ sub_end,
                      const uint16_t* __restrict__ sub_cnt, uint8_t* __restrict__ off, uint8_t* __restrict__ cnt) {
    const SyncTile t = tiles[blockIdx.x];
    const uint32_t end = (uint32_t)(8 + nbits[t.ss]);
    const uint32_t n_sub = (end + SUB_BITS - 1) / SUB_BITS;
    const uint32_t sub = t.sub0 + threadIdx.x;
    if (sub >= n_sub) return;
    const uint64_t g = t.sub_base + threadIdx.x;
    off[g] = sub == n_sub - 1 ? (uint8_t)0 : (uint8_t)(sub_end[g] - (sub + 1) * SUB_BITS);
    cnt[g] = (uint8_t)sub_cnt[g];
}

__global__ void __launch_bounds__(SUB_PER_CTA)
restart_load_kernel(const SyncTile* __restrict__ tiles, const uint64_t* __restrict__ nbits, const uint8_t* __restrict__ off,
                    const uint8_t* __restrict__ cnt, uint32_t* __restrict__ sub_end, uint16_t* __restrict__ sub_cnt,
                    uint32_t* __restrict__ tile_cnt) {
    __shared__ uint32_t s_red[SUB_PER_CTA / 32];
    const SyncTile t = tiles[blockIdx.x];
    const uint32_t end = (uint32_t)(8 + nbits[t.ss]);
    const uint32_t n_sub = (end + SUB_BITS - 1) / SUB_BITS;
    const uint32_t sub = t.sub0 + threadIdx.x;
    const bool active = sub < n_sub;
    const uint64_t g = t.sub_base + threadIdx.x;
    uint32_t v = 0;
    if (active) {
        v = cnt[g];
        sub_end[g] = sub == n_sub - 1 ? end : min(end, (sub + 1) * SUB_BITS + off[g]);
        sub_cnt[g] = (uint16_t)v;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t tot = 0;
        for (int w = 0; w < SUB_PER_CTA / 32; ++w) tot += s_red[w];
        tile_cnt[blockIdx.x] = tot;
    }
}

// The CTA's symbols are one contiguous run of the output, so they are staged in shared memory and
// written out coalesced (a thread's own run is only a few symbols long: writing it straight to global
// memory costs a 32-byte sector per 1- or 2-byte store).
constexpr int WRITE_STAGE = 10240;           // staged 16-bit symbols per CTA (twice as many of the byte-wide zero counts,
                                             // whose short codes put ~15 000 symbols into a tile); the rare overflow is written directly

__global__ void __launch_bounds__(SUB_PER_CTA)
huffman_write_kernel(SyncArgs a, Geom g, const uint32_t* __restrict__ tile_off, int16_t* __restrict__ dc,
                     int16_t* __restrict__ values, uint8_t* __restrict__ lengths, uint32_t* __restrict__ err) {
    extern __shared__ __align__(16) uint8_t write_raw[];
    uint32_t* s_words = reinterpret_cast<uint32_t*>(write_raw);
    int32_t* s_l1 = reinterpret_cast<int32_t*>(write_raw + 4 * (CHUNK_WORDS + CHUNK_SLACK));
    uint32_t* s_pk = reinterpret_cast<uint32_t*>(write_raw + 4 * (CHUNK_WORDS + CHUNK_SLACK) + 4 * L1_SIZE);
    int16_t* s_stage = reinterpret_cast<int16_t*>(write_raw + 4 * (CHUNK_WORDS + CHUNK_SLACK) + 4 * L1_SIZE + 4 * PK_SIZE);
    __shared__ uint32_t s_sum[SUB_PER_CTA / 32];
    __shared__ uint32_t s_staged;               // symbols [0, s_staged) of the CTA went through the staging area
    const SyncTile t = a.tiles[blockIdx.x];
    const uint32_t end = (uint32_t)(8 + a.nbits[t.ss]);
    const uint32_t n_sub = (end + SUB_BITS - 1) / SUB_BITS;
    const uint32_t sub = t.sub0 + threadIdx.x;
    const bool active = sub < n_sub;
    const uint64_t gi = t.sub_base + threadIdx.x;
    const uint32_t chunk0 = t.sub0 * SUB_BITS;
    if (threadIdx.x == 0) s_staged = 0xFFFFFFFFu;
    stage_chunk(a, t, s_words, s_l1);
    const bool packed = t.ss % 3 == HIC_KIND_LENGTH;     // byte-wide symbols, five per lookup
    const bool paired = t.ss % 3 == HIC_KIND_VALUE;      // two per lookup
    if (packed || paired) {
        const uint32_t* pk = a.pklut + ((size_t)(t.ss / 3) * 2 + (packed ? 1 : 0)) * PK_SIZE;
        for (int i = threadIdx.x; i < PK_SIZE; i += blockDim.x) s_pk[i] = __ldg(pk + i);
    }
    const BitReader br{s_words};
    const int32_t* l2 = a.lut2 + (size_t)t.ss * a.l2_cap;
    const RowIndex ridx = a.index[t.ss];
    const LongSearch ls{a.sorted_left + 2 * (size_t)ridx.offset, a.sorted_row + 2 * (size_t)ridx.offset,
                        a.row_sym + ridx.offset, a.row_packed + ridx.offset, ridx.count};
    const uint32_t cnt = active ? a.sub_cnt[gi] : 0;
    // exclusive scan of the counts inside the CTA
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = cnt;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const uint32_t o = __shfl_up_sync(0xffffffffu, inc, off);
        if (lane >= off) inc += o;
    }
    if (lane == 31) s_sum[warp] = inc;
    __syncthreads();            // also orders stage_chunk before the decode below
    uint32_t rank = inc - cnt, total = 0;
    for (int w = 0; w < SUB_PER_CTA / 32; ++w) {
        if (w < warp) rank += s_sum[w];
        total += s_sum[w];
    }
    const int img = t.ss / 9, c = (t.ss % 9) / 3, kind = t.ss % 3;
    const int64_t bb = cs_block_base(g, img, c);
    const uint32_t cap = (uint32_t)(kind == HIC_KIND_DC ? g.L.nb[c] : g.L.nb[c] * 64);
    const uint32_t tile_base = tile_off[blockIdx.x];
    const bool fits = tile_base + total <= cap;
    if (!fits && threadIdx.x == 0) atomicOr(err, 1u);
    int16_t* out16 = kind == HIC_KIND_DC ? dc + bb : values + bb * 64;
    uint8_t* out8 = kind == HIC_KIND_LENGTH ? lengths + bb * 64 : nullptr;
    if (active && fits) {
        const uint32_t start = sub == 0 ? 8u : a.sub_end[gi - 1];
        uint32_t got = 0;
        bool bad = false;
        uint32_t e;
        if (rank + cnt <= (uint32_t)(packed ? 2 * WRITE_STAGE : WRITE_STAGE)) {        // the usual case: into the staging area
            if (packed) e = decode_span_packed<uint8_t>(br, chunk0, start, (sub + 1) * SUB_BITS, end, s_l1, s_pk, l2, ls, got,
                                                        reinterpret_cast<uint8_t*>(s_stage), rank, bad);
            else if (paired) e = decode_span_packed<int16_t>(br, chunk0, start, (sub + 1) * SUB_BITS, end, s_l1, s_pk, l2, ls, got,
                                                             s_stage, rank, bad);
            else e = decode_span<true>(br, chunk0, start, (sub + 1) * SUB_BITS, end, s_l1, l2, ls, got, s_stage, nullptr, rank, bad);
        } else {                                          // ranks grow with the thread index: everything from here on is direct
            atomicMin(&s_staged, rank);
            e = decode_span<true>(br, chunk0, start, (sub + 1) * SUB_BITS, end, s_l1, l2, ls, got, out16, out8, tile_base + rank, bad);
        }
        if (bad || got != cnt || e != a.sub_end[gi] || (sub == n_sub - 1 && e != end)) atomicOr(err, 1u);
    }
    __syncthreads();
    if (!fits) return;
    const uint32_t staged = min(total, s_staged);
    if (out8) {
        const uint8_t* stage8 = reinterpret_cast<const uint8_t*>(s_stage);
        for (uint32_t i = threadIdx.x; i < staged; i += SUB_PER_CTA) out8[tile_base + i] = stage8[i];
    } else {
        for (uint32_t i = threadIdx.x; i < staged; i += SUB_PER_CTA) out16[tile_base + i] = s_stage[i];
    }
}

// ------------------------------------------------------------------------------------------------
// D2: run-length expansion.  position(i) = sum_{j<i} (len_j + 1) + len_i
// ------------------------------------------------------------------------------------------------
struct XRef {
    int img, c, tile;
};
__device__ __forceinline__ XRef locate(const int (&tiles)[3], int per_image, int64_t t) {
    XRef r;
    r.img = (int)(t / per_image);
    int rem = (int)(t - (int64_t)r.img * per_image);
    r.c = 0;
    while (rem >= tiles[r.c]) {
        rem -= tiles[r.c];
        ++r.c;
    }
    r.tile = rem;
    return r;
}

template <int THREADS>
__device__ __forceinline__ int64_t block_excl_sum64(int64_t v, int64_t* smem, int64_t* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int64_t inc = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int64_t o = __shfl_up_sync(0xffffffffu, inc, off);
        if (lane >= off) inc += o;
    }
    if (lane == 31) smem[warp] = inc;
    __syncthreads();
    int64_t base = 0, tot = 0;
    for (int w = 0; w < THREADS / 32; ++w) {
        if (w < warp) base += smem[w];
        tot += smem[w];
    }
    if (total) *total = tot;
    __syncthreads();
    return base + inc - v;
}

// positions covered by each tile of 2048 symbols: sum of (zero count + 1).  One WARP per tile (a lane
// reads four 16-byte vectors and adds their bytes with the SIMD absolute-difference instruction), eight
// tiles per CTA, no shared memory and no barrier: the grid covers the capacity, most of it empty tiles.
__global__ void __launch_bounds__(XTHREADS)
expand_tile_sum_kernel(Geom g, const uint8_t* __restrict__ lengths, const uint32_t* __restrict__ nsym_arr,
                       int64_t* __restrict__ tile_sum, int64_t total_tiles) {
    const int lane = threadIdx.x & 31;
    const int64_t t = (int64_t)blockIdx.x * (XTHREADS / 32) + (threadIdx.x >> 5);
    if (t >= total_tiles) return;
    const XRef r = locate(g.xtiles, g.xtiles_per_image, t);
    const int ss = (r.img * 3 + r.c) * 3 + HIC_KIND_LENGTH;
    const uint32_t nsym = nsym_arr[ss];
    const uint32_t tile_first = (uint32_t)r.tile * XT;
    uint32_t sum = 0;
    if (tile_first < nsym) {
        const uint32_t in_tile = min((uint32_t)XT, nsym - tile_first);
        const uint8_t* len = lengths + cs_block_base(g, r.img, r.c) * 64 + tile_first;      // 16-byte aligned
        static_assert(XT == 4 * 32 * 16, "four 16-byte vectors per lane");
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t off = (uint32_t)(j * 32 + lane) * 16u;
            if (off >= in_tile) continue;
            const uint4 v = *reinterpret_cast<const uint4*>(len + off);       // the symbol arrays carry slack past the end
            const uint32_t wv[4] = {v.x, v.y, v.z, v.w};
            const uint32_t valid = min(16u, in_tile - off);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t nb = valid > 4u * k ? min(4u, valid - 4u * k) : 0u;
                const uint32_t keep = nb == 4u ? 0xFFFFFFFFu : ((1u << (8u * nb)) - 1u);
                sum += __vsadu4(wv[k] & keep, 0u) + nb;
            }
        }
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) sum += __shfl_down_sync(0xffffffffu, sum, off);
    if (lane == 0) tile_sum[t] = (int64_t)sum;
}

// exclusive scan of the tile sums of every channel stream: one CTA per stream, SCAN_THREADS tiles at a time (a
// single huge image has three streams of tens of thousands of tiles: one thread walking them was 0.57 ms of an 8K
// wavelet decode)
constexpr int SCAN_THREADS = 256;
__global__ void __launch_bounds__(SCAN_THREADS)
stream_scan64_kernel(int n_cs, int tiles0, int tiles1, int tiles2, int per_image,
                     const int64_t* __restrict__ tile_sum, int64_t* __restrict__ tile_off,
                     int64_t* __restrict__ stream_total) {
    __shared__ long long s_warp[SCAN_THREADS / 32];
    const int cs = blockIdx.x;
    if (cs >= n_cs) return;
    const int img = cs / 3, c = cs % 3;
    const int tiles[3] = {tiles0, tiles1, tiles2};
    int64_t t0 = (int64_t)img * per_image;
    for (int k = 0; k < c; ++k) t0 += tiles[k];
    const int n = tiles[c];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long run = 0;
    for (int base = 0; base < n; base += SCAN_THREADS) {
        const int t = base + threadIdx.x;
        const long long v = t < n ? (long long)tile_sum[t0 + t] : 0ll;
        long long inc = v;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const long long o = __shfl_up_sync(0xffffffffu, inc, off);
            if (lane >= off) inc += o;
        }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        long long before = run;
        for (int k = 0; k < SCAN_THREADS / 32; ++k) {
            if (k < warp) before += s_warp[k];
            run += s_warp[k];
        }
        if (t < n) tile_off[t0 + t] = before + inc - v;
        __syncthreads();
    }
    if (threadIdx.x == 0) stream_total[cs] = run;
}

template <int THREADS>
__device__ __forceinline__ uint32_t block_excl_sum32(uint32_t v, uint32_t* smem, uint32_t* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const uint32_t o = __shfl_up_sync(0xffffffffu, inc, off);
        if (lane >= off) inc += o;
    }
    if (lane == 31) smem[warp] = inc;
    __syncthreads();
    uint32_t base = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < THREADS / 32; ++w) {
        if (w < warp) base += smem[w];
        tot += smem[w];
    }
    *total = tot;
    __syncthreads();
    return base + inc - v;
}

// Every tile of 2048 symbols owns the run of positions its symbols cover (at most 15 each).  The run is
// staged in shared memory in OUTPUT order -- zeros included, and in the block layout with the DC slot
// of every block it crosses (filled from the DC values dc_prefix_kernel has left, one int16 per block) --
// and leaves as 16-byte vectors; only the partial vectors at the two ends of the run go out element by
// element.  The tiles of a stream also share the zero tail behind the last symbol.  Every AC position
// is therefore written exactly once and the coefficient buffer needs no memset.
constexpr int XSTAGE = 8192;                 // staged output elements per pass (a tile covers <= 15 * XT positions)

__global__ void __launch_bounds__(XTHREADS)
expand_scatter_kernel(Geom g, const int16_t* __restrict__ values, const uint8_t* __restrict__ lengths,
                      const int16_t* __restrict__ dcval, const uint32_t* __restrict__ nsym_arr, const int64_t* __restrict__ tile_off,
                      const int64_t* __restrict__ stream_total, int16_t* __restrict__ coef, uint32_t* __restrict__ err) {
    __shared__ uint32_t s[XTHREADS / 32];
    __shared__ __align__(16) int16_t stage[XSTAGE];
    const XRef r = locate(g.xtiles, g.xtiles_per_image, blockIdx.x);
    const int cs = r.img * 3 + r.c;
    const uint32_t nsym = nsym_arr[cs * 3 + HIC_KIND_LENGTH];
    const int64_t bb = cs_block_base(g, r.img, r.c);
    const int64_t stream_len = g.L.len[r.c];
    int16_t* dst = coef + bb * 64;
    const bool skip = g.L.skip_first != 0;
    // DCT mode: element 0 of every block is its DC value (dc_prefix_kernel has turned the decoded differences
    // into values, one int16 per block).  A tile writes the DC slots inside its run of outputs, plus the one just
    // before it when its run starts a block; the zero tail writes those of the blocks it covers -- every DC slot
    // exactly once, and no separate pass of 2-byte stores into 128-byte lines (it moved 20x its bytes).
    const int16_t* dcs = dcval + bb;
    // positions fit 31 bits (hic_decode_plan_create): 32-bit arithmetic, division by the constant 63
    auto out_index = [&](uint32_t q) { return skip ? q + q / 63u + 1u : q; };
    const uint32_t tile_first = (uint32_t)r.tile * XT;
    if (tile_first < nsym) {
        const uint32_t start = tile_first + threadIdx.x * XSPT;
        static_assert(XSPT == 8, "one 8-byte and one 16-byte load per thread");
        uint32_t l[XSPT];
        int v[XSPT];
        uint32_t sum = 0;
        const uint32_t n_valid = start < nsym ? min((uint32_t)XSPT, nsym - start) : 0u;
        if (n_valid) {          // the symbol arrays carry slack: whole vectors may be read past the end
            const uint2 lv = *reinterpret_cast<const uint2*>(lengths + bb * 64 + start);
            const uint4 vv = *reinterpret_cast<const uint4*>(values + bb * 64 + start);
            const uint32_t vw[4] = {vv.x, vv.y, vv.z, vv.w};
#pragma unroll
            for (int j = 0; j < XSPT; ++j) {
                const bool in = (uint32_t)j < n_valid;
                l[j] = in ? ((j < 4 ? lv.x : lv.y) >> (8 * (j & 3))) & 0xFFu : 0u;
                v[j] = in ? (int)(short)((vw[j >> 1] >> (16 * (j & 1))) & 0xFFFF) : 0;
                sum += in ? l[j] + 1u : 0u;
            }
        } else {
#pragma unroll
            for (int j = 0; j < XSPT; ++j) {
                l[j] = 0;
                v[j] = 0;
            }
        }
        uint32_t tile_total;
        const uint32_t rank = block_excl_sum32<XTHREADS>(sum, s, &tile_total);
        const int64_t p0_64 = tile_off[blockIdx.x];
        if (p0_64 + tile_total > stream_len || tile_total == 0) {
            if (threadIdx.x == 0) atomicOr(err, 2u);
        } else {
            const uint32_t p0 = (uint32_t)p0_64;
            const uint32_t o_begin = out_index(p0) - ((skip && p0 % 63u == 0u) ? 1u : 0u), o_end = out_index(p0 + tile_total - 1u) + 1u;
            for (uint32_t base = o_begin & ~7u; base < o_end; base += XSTAGE) {
                const uint32_t span = min((uint32_t)XSTAGE, o_end - base);
                const uint32_t nvec = (span + 7u) >> 3;
                for (uint32_t i = threadIdx.x; i < nvec; i += XTHREADS) reinterpret_cast<uint4*>(stage)[i] = make_uint4(0, 0, 0, 0);
                __syncthreads();
                if (skip) {         // the DC slots of this pass (at most 128): one load per thread, all in flight together
                    for (uint32_t d = ((base + 63u) >> 6) + threadIdx.x; 64u * d < base + span; d += XTHREADS) stage[64u * d - base] = dcs[d];
                }
                uint32_t pos = p0 + rank;
#pragma unroll
                for (int j = 0; j < XSPT; ++j) {
                    const uint32_t q = out_index(pos + l[j]) - base;       // wraps below `base`: fails the bound check
                    if (v[j] != 0 && q < span) stage[q] = (int16_t)v[j];
                    pos += (uint32_t)j < n_valid ? l[j] + 1u : 0u;
                }
                __syncthreads();
                for (uint32_t i = threadIdx.x; i < nvec; i += XTHREADS) {
                    const uint32_t o = base + 8u * i;
                    if (o >= o_begin && o + 8u <= o_end) {
                        *reinterpret_cast<uint4*>(dst + o) = reinterpret_cast<const uint4*>(stage)[i];
                    } else {
#pragma unroll
                        for (uint32_t k = 0; k < 8u; ++k)
                            if (o + k >= o_begin && o + k < o_end) dst[o + k] = stage[8u * i + k];
                    }
                }
                __syncthreads();
            }
        }
    }
    // the zero tail behind the stream's last symbol, split over the stream's tiles
    const int64_t tail0 = min(stream_total[cs], stream_len);
    const int64_t share = (stream_len - tail0 + g.xtiles[r.c] - 1) / g.xtiles[r.c];
    const int64_t a = tail0 + share * r.tile, b = min(stream_len, a + share);
    for (int64_t p = a + threadIdx.x; p < b; p += XTHREADS) {
        if (skip) {
            const uint32_t q = (uint32_t)p, blk = q / 63u;
            dst[q + blk + 1u] = 0;
            if (q == 63u * blk) dst[64u * blk] = dcs[blk];
        } else {
            dst[p] = 0;
        }
    }
}

// validates each channel stream's expanded length (codec.py:109-111: only a trailing (0,0) may
// leave the array short) and the symbol counts
__global__ void validate_kernel(Geom g, const int16_t* __restrict__ values, const uint8_t* __restrict__ lengths,
                                const uint32_t* __restrict__ nsym_arr, const int64_t* __restrict__ stream_total,
                                uint32_t* __restrict__ err) {
    const int cs = blockIdx.x * blockDim.x + threadIdx.x;
    if (cs >= g.L.n_images * 3) return;
    const int img = cs / 3, c = cs % 3;
    const uint32_t n_val = nsym_arr[cs * 3 + HIC_KIND_VALUE], n_len = nsym_arr[cs * 3 + HIC_KIND_LENGTH];
    if (n_val != n_len || n_len == 0) {
        atomicOr(err, 4u);
        return;
    }
    if (g.L.skip_first && nsym_arr[cs * 3 + HIC_KIND_DC] != (uint32_t)g.L.nb[c]) atomicOr(err, 8u);
    const int64_t bb = cs_block_base(g, img, c);
    const bool trailing = values[bb * 64 + n_len - 1] == 0 && lengths[bb * 64 + n_len - 1] == 0;
    const int64_t total = stream_total[cs];
    if (trailing ? (total > g.L.len[c]) : (total != g.L.len[c])) atomicOr(err, 16u);
}

// the DC-only decode's check: every DC stream held exactly one symbol per block of its channel
__global__ void validate_dc_kernel(Geom g, const uint32_t* __restrict__ nsym_arr, uint32_t* __restrict__ err) {
    const int cs = blockIdx.x * blockDim.x + threadIdx.x;
    if (cs >= g.L.n_images * 3) return;
    if (nsym_arr[cs * 3 + HIC_KIND_DC] != (uint32_t)g.L.nb[cs % 3]) atomicOr(err, 8u);
}

// ------------------------------------------------------------------------------------------------
// D3: DC prefix sum (utils.invert_differences) written to element 0 of every block
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(XTHREADS)
dc_tile_sum_kernel(Geom g, const int16_t* __restrict__ dc, int64_t* __restrict__ tile_sum) {
    __shared__ int64_t s[XTHREADS / 32];
    const XRef r = locate(g.dtiles, g.dtiles_per_image, blockIdx.x);
    const int64_t nb = g.L.nb[r.c];
    const int16_t* src = dc + cs_block_base(g, r.img, r.c);
    const int64_t start = (int64_t)r.tile * XT + threadIdx.x * XSPT;
    int64_t sum = 0;
#pragma unroll
    for (int j = 0; j < XSPT; ++j)
        if (start + j < nb) sum += src[start + j];
    int64_t total;
    block_excl_sum64<XTHREADS>(sum, s, &total);
    if (threadIdx.x == 0) tile_sum[blockIdx.x] = total;
}

// the decoded DC differences of every channel stream become DC values in place (one int16 per block)
__global__ void __launch_bounds__(XTHREADS)
dc_prefix_kernel(Geom g, int16_t* __restrict__ dc, const int64_t* __restrict__ tile_off) {
    __shared__ int64_t s[XTHREADS / 32];
    const XRef r = locate(g.dtiles, g.dtiles_per_image, blockIdx.x);
    const int64_t nb = g.L.nb[r.c];
    int16_t* src = dc + cs_block_base(g, r.img, r.c);
    const int64_t start = (int64_t)r.tile * XT + threadIdx.x * XSPT;
    int d[XSPT];
    int64_t sum = 0;
#pragma unroll
    for (int j = 0; j < XSPT; ++j) {
        d[j] = start + j < nb ? src[start + j] : 0;
        sum += d[j];
    }
    int64_t run = tile_off[blockIdx.x] + block_excl_sum64<XTHREADS>(sum, s, nullptr);
#pragma unroll
    for (int j = 0; j < XSPT; ++j) {
        if (start + j >= nb) break;
        run += d[j];
        src[start + j] = (int16_t)run;
    }
}

}  // namespace dec
}  // namespace hic

using namespace hic;
using namespace hic::dec;

struct hic_decode_plan {
    dec::Geom g;
    int n_cs = 0, n_ss = 0;
    int64_t total_blocks = 0, total_xtiles = 0, total_dtiles = 0;
    int16_t* d_dc = nullptr;
    int16_t* d_values = nullptr;
    uint8_t* d_lengths = nullptr;
    int32_t* d_lut1 = nullptr;
    int32_t* d_lut2 = nullptr;
    uint16_t* d_mlut = nullptr;                 // multi-symbol table of the sync passes
    uint32_t* d_pklut = nullptr;                // packed multi-symbol tables per channel stream: [0] value pairs, [1] zero counts
    int l2_cap = L2_CAP_MIN;
    uint64_t* d_sorted_left = nullptr;          // 2 x row capacity (bitonic padding)
    uint32_t* d_sorted_row = nullptr;
    uint64_t sorted_capacity = 0;
    SyncTile* d_tiles = nullptr;
    uint64_t tile_capacity = 0;
    uint32_t* d_ss_tile0 = nullptr;
    uint32_t* d_sub_end = nullptr;
    uint16_t* d_sub_cnt = nullptr;
    uint64_t sub_capacity = 0;
    uint8_t* d_restart = nullptr;               // 2 x sub_capacity: `off` bytes then `cnt` bytes of the restart records
    uint64_t data_bytes = 0;                    // size of the caller's d_bytes buffer when it said so (0: unknown, not checked)
    uint64_t last_n_sub = 0, last_n_tiles = 0;  // of the most recent run (what hic_decode_export_restarts exports)
    uint32_t* d_tile_start = nullptr;
    uint32_t* d_tile_cnt = nullptr;
    uint32_t* d_tile_symoff = nullptr;
    RowIndex* d_index_own = nullptr;            // tables uploaded from the host live in the plan ...
    int32_t* d_row_sym_own = nullptr;
    uint64_t* d_row_packed_own = nullptr;
    uint64_t row_capacity = 0;
    const RowIndex* d_index = nullptr;          // ... tables handed over on the device are only referenced
    const int32_t* d_row_sym = nullptr;
    const uint64_t* d_row_packed = nullptr;
    uint64_t* d_byte_off = nullptr;
    uint64_t* d_nbits = nullptr;
    uint32_t* d_nsym = nullptr;
    uint32_t* d_err = nullptr;
    int64_t* d_tile_sum = nullptr;
    int64_t* d_tile_off = nullptr;
    int64_t* d_stream_total = nullptr;
    bool tables_ready = false;
    hic::SmallXfer xfer;                        // page-locked staging of the small transfers (reset after every synchronisation)
};

template <typename T>
static cudaError_t dalloc2(T** p, size_t count) {
    return cudaMalloc(reinterpret_cast<void**>(p), (count ? count : 1) * sizeof(T));
}

extern "C" {

int hic_decode_plan_destroy(hic_decode_plan* p) {
    if (!p) return HIC_OK;
    p->xfer.destroy();
    void* ptrs[] = {p->d_restart, p->d_pklut, p->d_mlut, p->d_dc, p->d_values, p->d_lengths, p->d_lut1, p->d_lut2, p->d_sorted_left, p->d_sorted_row, p->d_tiles, p->d_ss_tile0, p->d_sub_end,
                    p->d_sub_cnt, p->d_tile_start, p->d_tile_cnt, p->d_tile_symoff, p->d_index_own, p->d_row_sym_own,
                    p->d_row_packed_own, p->d_byte_off, p->d_nbits, p->d_nsym, p->d_err, p->d_tile_sum,
                    p->d_tile_off, p->d_stream_total};
    for (void* q : ptrs)
        if (q) cudaFree(q);
    delete p;
    return HIC_OK;
}

int hic_decode_plan_create(const hic_stream_layout* L, hic_decode_plan** out) {
    HIC_REQUIRE(out != nullptr && L != nullptr, "NULL argument");
    *out = nullptr;
    HIC_REQUIRE(L->n_images >= 1, "layout has no images");
    hic_decode_plan* p = new hic_decode_plan();
    p->g.L = *L;
    p->g.xtiles_per_image = p->g.dtiles_per_image = 0;
    for (int c = 0; c < 3; ++c) {
        if (L->nb[c] < 1 || L->nb[c] * 64 >= (1ll << 31)) {
            delete p;
            return hic::fail(HIC_ERR_INVALID, "channel stream too long");
        }
        p->g.xtiles[c] = (int)((L->nb[c] * 64 + XT - 1) / XT);
        p->g.dtiles[c] = L->skip_first ? (int)((L->nb[c] + XT - 1) / XT) : 0;
        p->g.xtiles_per_image += p->g.xtiles[c];
        p->g.dtiles_per_image += p->g.dtiles[c];
    }
    p->n_cs = L->n_images * 3;
    p->n_ss = L->n_images * 9;
    p->total_blocks = (int64_t)L->n_images * L->blocks_per_image;
    p->total_xtiles = (int64_t)L->n_images * p->g.xtiles_per_image;
    p->total_dtiles = (int64_t)L->n_images * p->g.dtiles_per_image;
    cudaError_t e = cudaSuccess;
    auto ok = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
    ok(dalloc2(&p->d_dc, p->total_blocks));
    ok(dalloc2(&p->d_values, p->total_blocks * 64 + 64));
    ok(dalloc2(&p->d_lengths, p->total_blocks * 64 + 64));
    ok(dalloc2(&p->d_lut1, (size_t)p->n_ss * L1_SIZE));
    ok(dalloc2(&p->d_mlut, (size_t)p->n_ss * L1_SIZE));
    ok(dalloc2(&p->d_pklut, (size_t)p->n_cs * 2 * PK_SIZE));
    {
        int cap = L2_CAP_MAX;
        while (cap > L2_CAP_MIN && (size_t)cap * p->n_ss > ((size_t)1 << 28)) cap >>= 1;
        p->l2_cap = cap;
    }
    ok(dalloc2(&p->d_lut2, (size_t)p->n_ss * p->l2_cap));
    ok(dalloc2(&p->d_ss_tile0, p->n_ss + 1));
    ok(dalloc2(&p->d_index_own, p->n_ss));
    ok(dalloc2(&p->d_byte_off, p->n_ss));
    ok(dalloc2(&p->d_nbits, p->n_ss));
    ok(dalloc2(&p->d_nsym, p->n_ss));
    ok(dalloc2(&p->d_err, 4));
    ok(dalloc2(&p->d_tile_sum, std::max(p->total_xtiles, p->total_dtiles)));
    ok(dalloc2(&p->d_tile_off, std::max(p->total_xtiles, p->total_dtiles)));
    ok(dalloc2(&p->d_stream_total, p->n_cs));
    if (e != cudaSuccess) {
        hic_decode_plan_destroy(p);
        return hic::fail(HIC_ERR_CUDA, "decode plan allocation failed: %s", cudaGetErrorString(e));
    }
    *out = p;
    return HIC_OK;
}

int hic_decode_set_tables_device(hic_decode_plan* p, const void* d_index, const int32_t* d_row_sym,
                                 const uint64_t* d_row_packed, uint64_t total_rows, void* stream) {
    HIC_REQUIRE(p && d_index && d_row_sym && d_row_packed, "NULL argument");
    cudaStream_t st = as_stream(stream);
    p->d_index = static_cast<const RowIndex*>(d_index);
    p->d_row_sym = d_row_sym;
    p->d_row_packed = d_row_packed;
    if (total_rows > p->sorted_capacity) {          // scratch for the long-code search (2x: bitonic padding)
        HIC_CUDA(cudaStreamSynchronize(st));
        if (p->d_sorted_left) cudaFree(p->d_sorted_left);
        if (p->d_sorted_row) cudaFree(p->d_sorted_row);
        p->d_sorted_left = nullptr; p->d_sorted_row = nullptr;
        p->sorted_capacity = total_rows + total_rows / 4 + 1024;
        HIC_CUDA(dalloc2(&p->d_sorted_left, 2 * p->sorted_capacity));
        HIC_CUDA(dalloc2(&p->d_sorted_row, 2 * p->sorted_capacity));
    }
    HIC_LAUNCH("build_tables_kernel", st, build_tables_kernel<<<p->n_ss, 256, 0, st>>>(p->d_index, p->d_row_sym, p->d_row_packed, p->d_lut1, p->d_lut2,
                                                                                         p->l2_cap, p->d_sorted_left, p->d_sorted_row, p->d_mlut, p->d_pklut));
    p->tables_ready = true;
    return HIC_OK;
}

int hic_decode_set_tables_packed(hic_decode_plan* p, const uint32_t* h_index, const int32_t* h_row_sym,
                                 const uint64_t* h_row_packed, uint64_t total, void* stream) {
    HIC_REQUIRE(p && h_index && h_row_sym && h_row_packed, "NULL argument");
    HIC_REQUIRE(total < (1ull << 32), "too many table rows");
    cudaStream_t st = as_stream(stream);
    for (int s = 0; s < p->n_ss; ++s)
        HIC_REQUIRE((uint64_t)h_index[2 * s] + h_index[2 * s + 1] <= total, "stream %d: rows [%u, +%u) exceed %llu", s,
                    h_index[2 * s], h_index[2 * s + 1], (unsigned long long)total);
    if (total > p->row_capacity) {
        if (p->d_row_sym_own) cudaFree(p->d_row_sym_own);
        if (p->d_row_packed_own) cudaFree(p->d_row_packed_own);
        p->d_row_sym_own = nullptr; p->d_row_packed_own = nullptr;
        p->row_capacity = total + total / 4 + 1024;
        HIC_CUDA(dalloc2(&p->d_row_sym_own, p->row_capacity));
        HIC_CUDA(dalloc2(&p->d_row_packed_own, p->row_capacity));
    }
    static_assert(sizeof(RowIndex) == 2 * sizeof(uint32_t), "index layout");
    // (through the SMs when the caller's arrays are page-locked: see SmallXfer)
    int rc = hic::small_h2d(p->xfer, p->d_index_own, h_index, sizeof(RowIndex) * p->n_ss, st);
    if (rc) return rc;
    if (total) {
        rc = hic::small_h2d(p->xfer, p->d_row_sym_own, h_row_sym, sizeof(int32_t) * total, st);
        if (rc) return rc;
        rc = hic::small_h2d(p->xfer, p->d_row_packed_own, h_row_packed, sizeof(uint64_t) * total, st);
        if (rc) return rc;
    }
    return hic_decode_set_tables_device(p, p->d_index_own, p->d_row_sym_own ? p->d_row_sym_own : (const int32_t*)p->d_index_own,
                                        p->d_row_packed_own ? p->d_row_packed_own : (const uint64_t*)p->d_index_own, total, stream);
}

int hic_decode_set_tables(hic_decode_plan* p, const uint32_t* h_rows, const int32_t* h_symbols, const uint8_t* h_lens,
                          const uint64_t* h_codes, void* stream) {
    HIC_REQUIRE(p && h_rows && h_symbols && h_lens && h_codes, "NULL argument");
    cudaStream_t st = as_stream(stream);
    const int nss = p->n_ss;
    std::vector<RowIndex> index(nss);
    uint64_t total = 0;
    for (int s = 0; s < nss; ++s) {
        HIC_REQUIRE(total + h_rows[s] < (1ull << 32), "too many table rows");
        index[s] = RowIndex{(uint32_t)total, h_rows[s]};
        total += h_rows[s];
    }
    std::vector<uint64_t> packed(total);
    for (uint64_t r = 0; r < total; ++r) {
        HIC_REQUIRE(h_lens[r] >= 1 && h_lens[r] <= 58, "code length %u out of range in row %llu", (unsigned)h_lens[r],
                    (unsigned long long)r);
        packed[r] = ((uint64_t)h_lens[r] << 58) | (h_codes[r] & ((1ull << 58) - 1));
    }
    if (total > p->row_capacity) {
        if (p->d_row_sym_own) cudaFree(p->d_row_sym_own);
        if (p->d_row_packed_own) cudaFree(p->d_row_packed_own);
        p->d_row_sym_own = nullptr; p->d_row_packed_own = nullptr;
        p->row_capacity = total + total / 4 + 1024;
        HIC_CUDA(dalloc2(&p->d_row_sym_own, p->row_capacity));
        HIC_CUDA(dalloc2(&p->d_row_packed_own, p->row_capacity));
    }
    HIC_CUDA(cudaMemcpyAsync(p->d_index_own, index.data(), sizeof(RowIndex) * nss, cudaMemcpyHostToDevice, st));
    if (total) {
        HIC_CUDA(cudaMemcpyAsync(p->d_row_sym_own, h_symbols, sizeof(int32_t) * total, cudaMemcpyHostToDevice, st));
        HIC_CUDA(cudaMemcpyAsync(p->d_row_packed_own, packed.data(), sizeof(uint64_t) * total, cudaMemcpyHostToDevice, st));
    }
    int rc = hic_decode_set_tables_device(p, p->d_index_own, p->d_row_sym_own ? p->d_row_sym_own : (const int32_t*)p->d_index_own,
                                          p->d_row_packed_own ? p->d_row_packed_own : (const uint64_t*)p->d_index_own, total, stream);
    if (rc) return rc;
    HIC_CUDA(cudaStreamSynchronize(st));      // the staging vectors go out of scope
    return HIC_OK;
}

}  // extern "C"

// mode 0: the whole decode; mode 1: D1's synchronisation only (what the restart records are exported from);
// mode 2: the DC streams alone -- D1 on the kind-0 streams and D3 into d_coef, which is then one int16 DC value
// per block (the other streams' offsets and bit counts are ignored, their bytes never read);
// h_roff / h_rcnt: restart records of every subsequence in stream order (of the decoded streams), or NULL
static int decode_run_impl(hic_decode_plan* p, const uint8_t* d_bytes, const uint64_t* h_byte_off, const uint64_t* h_nbits,
                           int16_t* d_coef, void* stream, int mode, const uint8_t* h_roff, const uint8_t* h_rcnt,
                           uint64_t n_restart) {
    HIC_REQUIRE(p && d_bytes && h_byte_off && h_nbits && (d_coef || mode == 1), "NULL argument");
    // whatever way this call ends, the staging area of the small transfers is free again for the next one (an
    // early return used to leave it filled: after a few failed calls every small_d2h returned HIC_ERR_CAPACITY)
    struct XferGuard {
        hic::SmallXfer& x;
        cudaStream_t st;
        ~XferGuard() {
            cudaStreamSynchronize(st);          // nothing in flight reads or writes the staging any more
            x.reset();
        }
    } xfer_guard{p->xfer, as_stream(stream)};
    HIC_REQUIRE(p->tables_ready, "hic_decode_set_tables has not run");
    HIC_REQUIRE((reinterpret_cast<uintptr_t>(d_bytes) & 3) == 0, "d_bytes must be 4-byte aligned");
    const dec::Geom& g = p->g;
    cudaStream_t st = as_stream(stream);
    const int nss = p->n_ss;
    if (mode == 2) HIC_REQUIRE(g.L.skip_first, "a flat (wavelet) layout has no DC streams");
    std::vector<uint64_t> nbits(nss), off(nss);
    for (int s = 0; s < nss; ++s) {
        const bool used = mode != 2 || s % 3 == HIC_KIND_DC;
        nbits[s] = used ? h_nbits[s] : 0;
        off[s] = used ? h_byte_off[s] : 0;
        HIC_REQUIRE((off[s] & 3) == 0, "stream %d is not 4-byte aligned", s);
        // a framed payload is its pad-count byte + ceil(nbits / 8) bytes; the decoders read whole 32-bit words of it
        if (p->data_bytes && nbits[s])
            HIC_REQUIRE(off[s] + 4 * ((8 + nbits[s] + 31) / 32) <= p->data_bytes,
                        "stream %d (%llu bits at byte %llu) runs past the %llu bytes of d_bytes", s, (unsigned long long)nbits[s],
                        (unsigned long long)off[s], (unsigned long long)p->data_bytes);
    }
    {
        int rc = hic::small_h2d(p->xfer, p->d_byte_off, off.data(), sizeof(uint64_t) * nss, st);
        if (rc) return rc;
        rc = hic::small_h2d(p->xfer, p->d_nbits, nbits.data(), sizeof(uint64_t) * nss, st);
        if (rc) return rc;
    }
    HIC_CUDA(cudaMemsetAsync(p->d_err, 0, 4 * sizeof(uint32_t), st));
    // ---- D1: tiles of SUB_PER_CTA subsequences, streams in order ----
    std::vector<SyncTile> tiles;
    std::vector<uint32_t> ss_tile0(nss + 1, 0);
    uint64_t n_sub_total = 0;
    for (int s = 0; s < nss; ++s) {
        ss_tile0[s] = (uint32_t)tiles.size();
        if (nbits[s] == 0) continue;
        HIC_REQUIRE(nbits[s] + 8 < (1ull << 32), "stream %d too long", s);
        const uint64_t n_sub = (8 + nbits[s] + SUB_BITS - 1) / SUB_BITS;
        for (uint64_t sub0 = 0; sub0 < n_sub; sub0 += SUB_PER_CTA)
            tiles.push_back(SyncTile{(uint32_t)s, (uint32_t)sub0, n_sub_total + sub0});
        n_sub_total += n_sub;
    }
    ss_tile0[nss] = (uint32_t)tiles.size();
    const uint64_t n_tiles = tiles.size();
    if (n_tiles > p->tile_capacity) {
        for (void* q : {(void*)p->d_tiles, (void*)p->d_tile_start, (void*)p->d_tile_cnt, (void*)p->d_tile_symoff})
            if (q) cudaFree(q);
        p->d_tiles = nullptr; p->d_tile_start = nullptr; p->d_tile_cnt = nullptr; p->d_tile_symoff = nullptr;
        p->tile_capacity = n_tiles + n_tiles / 4 + 64;
        HIC_CUDA(dalloc2(&p->d_tiles, p->tile_capacity));
        HIC_CUDA(dalloc2(&p->d_tile_start, p->tile_capacity));
        HIC_CUDA(dalloc2(&p->d_tile_cnt, p->tile_capacity));
        HIC_CUDA(dalloc2(&p->d_tile_symoff, p->tile_capacity));
    }
    if (n_sub_total > p->sub_capacity) {
        if (p->d_sub_end) cudaFree(p->d_sub_end);
        if (p->d_sub_cnt) cudaFree(p->d_sub_cnt);
        if (p->d_restart) cudaFree(p->d_restart);
        p->d_sub_end = nullptr; p->d_sub_cnt = nullptr; p->d_restart = nullptr;
        p->sub_capacity = n_sub_total + n_sub_total / 4 + 1024;
        HIC_CUDA(dalloc2(&p->d_sub_end, p->sub_capacity));
        HIC_CUDA(dalloc2(&p->d_sub_cnt, p->sub_capacity));
        HIC_CUDA(dalloc2(&p->d_restart, 2 * p->sub_capacity));
    }
    p->last_n_sub = n_sub_total;
    p->last_n_tiles = n_tiles;
    const bool restarts = h_roff != nullptr;
    if (restarts) {
        HIC_REQUIRE(h_rcnt != nullptr && n_restart == n_sub_total, "restart records for %llu subsequences, the streams have %llu",
                    (unsigned long long)n_restart, (unsigned long long)n_sub_total);
    }
    {
        int rc = hic::small_h2d(p->xfer, p->d_ss_tile0, ss_tile0.data(), sizeof(uint32_t) * (nss + 1), st);
        if (rc) return rc;
    }
    HIC_CUDA(cudaMemsetAsync(p->d_nsym, 0, sizeof(uint32_t) * nss, st));
    int16_t* const dc = mode == 2 ? d_coef : p->d_dc;      // the DC-only mode decodes straight into the caller's buffer
    if (n_tiles) {
        {
            int rc = hic::small_h2d(p->xfer, p->d_tiles, tiles.data(), sizeof(SyncTile) * n_tiles, st);
            if (rc) return rc;
        }
        SyncArgs a;
        a.bytes = d_bytes; a.byte_off = p->d_byte_off; a.nbits = p->d_nbits; a.lut1 = p->d_lut1; a.lut2 = p->d_lut2; a.mlut = p->d_mlut; a.pklut = p->d_pklut; a.l2_cap = p->l2_cap; a.sorted_left = p->d_sorted_left; a.sorted_row = p->d_sorted_row;
        a.index = p->d_index; a.row_sym = p->d_row_sym; a.row_packed = p->d_row_packed; a.tiles = p->d_tiles; a.sub_end = p->d_sub_end;
        a.sub_cnt = p->d_sub_cnt; a.tile_start = p->d_tile_start; a.tile_cnt = p->d_tile_cnt; a.changed = p->d_err + 1;
        if (restarts) {
            HIC_CUDA(cudaMemcpyAsync(p->d_restart, h_roff, n_sub_total, cudaMemcpyHostToDevice, st));
            HIC_CUDA(cudaMemcpyAsync(p->d_restart + p->sub_capacity, h_rcnt, n_sub_total, cudaMemcpyHostToDevice, st));
            HIC_LAUNCH("restart_load_kernel", st, restart_load_kernel<<<(unsigned)n_tiles, SUB_PER_CTA, 0, st>>>(p->d_tiles, p->d_nbits, p->d_restart,
                                                                  p->d_restart + p->sub_capacity, p->d_sub_end, p->d_sub_cnt, p->d_tile_cnt));
        } else {
            HIC_LAUNCH("huffman_sync_kernel", st, huffman_sync_kernel<false><<<(unsigned)n_tiles, SUB_PER_CTA, 0, st>>>(a));
        }
        // A resynchronisation round carries a correction across at least one tile boundary, so a stream of T tiles
        // is settled after at most T rounds (codes that never self-synchronise -- complete trees of equal code
        // length 3, 5, 6 or 7, whose codewords straddle the 128-bit subsequences -- need them all).  More rounds
        // than the longest stream has tiles means the passes are not converging: that is reported as such, not as
        // a corrupt stream.
        uint64_t max_tiles_per_stream = 1;
        for (int s = 0; s < nss; ++s) max_tiles_per_stream = std::max<uint64_t>(max_tiles_per_stream, ss_tile0[s + 1] - ss_tile0[s]);
        bool settled = restarts;
        for (uint64_t round = 0; round <= max_tiles_per_stream && !settled; ++round) {
            HIC_CUDA(cudaMemsetAsync(p->d_err + 1, 0, sizeof(uint32_t), st));
            HIC_LAUNCH("huffman_resync_kernel", st, huffman_sync_kernel<true><<<(unsigned)n_tiles, SUB_PER_CTA, 0, st>>>(a));
            const void* h_changed = nullptr;
            {
                int rc = hic::small_d2h(p->xfer, p->d_err + 1, sizeof(uint32_t), st, &h_changed);
                if (rc) return rc;
            }
            HIC_CUDA(cudaStreamSynchronize(st));
            p->xfer.reset();
            if (!*static_cast<const volatile uint32_t*>(h_changed)) settled = true;
        }
        if (!settled)
            return hic::fail(HIC_ERR_INVALID, "the Huffman synchronisation passes did not settle within %llu rounds (the longest stream has "
                                              "that many tiles): not a corrupt stream, a decoder fault",
                             (unsigned long long)max_tiles_per_stream + 1);
        HIC_LAUNCH("sync_tile_scan_kernel", st, sync_tile_scan_kernel<<<(nss + 127) / 128, 128, 0, st>>>(nss, p->d_ss_tile0, p->d_tile_cnt, p->d_tile_symoff, p->d_nsym));
        if (mode == 1) {
            HIC_CUDA(cudaStreamSynchronize(st));
            p->xfer.reset();
            return HIC_OK;
        }
        {
            constexpr int WRITE_SMEM = 4 * (CHUNK_WORDS + CHUNK_SLACK) + 4 * L1_SIZE + 4 * PK_SIZE + 2 * WRITE_STAGE;
            static bool attr_set[64] = {false};
            int dev = 0;
            HIC_CUDA(cudaGetDevice(&dev));
            if (dev >= 64 || !attr_set[dev]) {
                HIC_CUDA(cudaFuncSetAttribute(huffman_write_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, WRITE_SMEM));
                if (dev < 64) attr_set[dev] = true;
            }
            HIC_LAUNCH("huffman_write_kernel", st, huffman_write_kernel<<<(unsigned)n_tiles, SUB_PER_CTA, WRITE_SMEM, st>>>(a, g, p->d_tile_symoff, dc, p->d_values, p->d_lengths, p->d_err));
        }
    }
    if (mode == 1) {
        HIC_CUDA(cudaStreamSynchronize(st));
        p->xfer.reset();
        return HIC_OK;
    }
    if (g.L.skip_first) {           // D3 first: the expansion below writes the DC values with the blocks they belong to
        HIC_LAUNCH("dc_tile_sum_kernel", st, dc_tile_sum_kernel<<<(unsigned)p->total_dtiles, XTHREADS, 0, st>>>(g, dc, p->d_tile_sum));
        HIC_LAUNCH("stream_scan64_kernel", st, stream_scan64_kernel<<<p->n_cs, SCAN_THREADS, 0, st>>>(p->n_cs, g.dtiles[0], g.dtiles[1], g.dtiles[2],
                                                                   g.dtiles_per_image, p->d_tile_sum, p->d_tile_off,
                                                                   p->d_stream_total));
        HIC_LAUNCH("dc_prefix_kernel", st, dc_prefix_kernel<<<(unsigned)p->total_dtiles, XTHREADS, 0, st>>>(g, dc, p->d_tile_off));
    }
    if (mode == 2) {
        HIC_LAUNCH("validate_dc_kernel", st, validate_dc_kernel<<<(p->n_cs + 127) / 128, 128, 0, st>>>(g, p->d_nsym, p->d_err));
    } else {
        HIC_LAUNCH("expand_tile_sum_kernel", st, expand_tile_sum_kernel<<<(unsigned)((p->total_xtiles + XTHREADS / 32 - 1) / (XTHREADS / 32)), XTHREADS, 0, st>>>(g, p->d_lengths, p->d_nsym, p->d_tile_sum, p->total_xtiles));
        HIC_LAUNCH("stream_scan64_kernel", st, stream_scan64_kernel<<<p->n_cs, SCAN_THREADS, 0, st>>>(p->n_cs, g.xtiles[0], g.xtiles[1], g.xtiles[2],
                                                                   g.xtiles_per_image, p->d_tile_sum, p->d_tile_off,
                                                                   p->d_stream_total));
        HIC_LAUNCH("expand_scatter_kernel", st, expand_scatter_kernel<<<(unsigned)p->total_xtiles, XTHREADS, 0, st>>>(g, p->d_values, p->d_lengths, p->d_dc, p->d_nsym,
                                                                             p->d_tile_off, p->d_stream_total, d_coef, p->d_err));
        HIC_LAUNCH("validate_kernel", st, validate_kernel<<<(p->n_cs + 127) / 128, 128, 0, st>>>(g, p->d_values, p->d_lengths, p->d_nsym, p->d_stream_total, p->d_err));
    }
    const void* h_flags = nullptr;
    {
        int rc = hic::small_d2h(p->xfer, p->d_err, 4 * sizeof(uint32_t), st, &h_flags);
        if (rc) return rc;
    }
    HIC_CUDA(cudaStreamSynchronize(st));
    const uint32_t flags0 = static_cast<const volatile uint32_t*>(h_flags)[0];
    p->xfer.reset();                 // everything staged has been consumed
    if (flags0) return hic::fail(HIC_ERR_CORRUPT, "bit streams did not decode cleanly (flags 0x%x)%s", flags0,
                                 restarts ? " -- or the restart records do not belong to them" : "");
    return HIC_OK;
}

extern "C" {

int hic_decode_set_data_bytes(hic_decode_plan* p, uint64_t nbytes) {
    HIC_REQUIRE(p != nullptr, "plan is NULL");
    p->data_bytes = nbytes;
    return HIC_OK;
}

int hic_decode_run(hic_decode_plan* p, const uint8_t* d_bytes, const uint64_t* h_byte_off, const uint64_t* h_nbits,
                   int16_t* d_coef, void* stream) {
    return decode_run_impl(p, d_bytes, h_byte_off, h_nbits, d_coef, stream, 0, nullptr, nullptr, 0);
}

int hic_decode_run_restarts(hic_decode_plan* p, const uint8_t* d_bytes, const uint64_t* h_byte_off, const uint64_t* h_nbits,
                            const uint8_t* h_off, const uint8_t* h_cnt, uint64_t n_sub, int16_t* d_coef, void* stream) {
    HIC_REQUIRE(h_off && h_cnt, "NULL restart records");
    return decode_run_impl(p, d_bytes, h_byte_off, h_nbits, d_coef, stream, 0, h_off, h_cnt, n_sub);
}

int hic_decode_run_dc(hic_decode_plan* p, const uint8_t* d_bytes, const uint64_t* h_byte_off, const uint64_t* h_nbits,
                      const uint8_t* h_off, const uint8_t* h_cnt, uint64_t n_sub, int16_t* d_dc, void* stream) {
    HIC_REQUIRE((h_off == nullptr) == (h_cnt == nullptr), "restart records need both `off` and `cnt`");
    return decode_run_impl(p, d_bytes, h_byte_off, h_nbits, d_dc, stream, 2, h_off, h_cnt, n_sub);
}

int hic_decode_sync(hic_decode_plan* p, const uint8_t* d_bytes, const uint64_t* h_byte_off, const uint64_t* h_nbits,
                    uint64_t* n_sub_out, void* stream) {
    const int rc = decode_run_impl(p, d_bytes, h_byte_off, h_nbits, nullptr, stream, 1, nullptr, nullptr, 0);
    if (rc) return rc;
    if (n_sub_out) *n_sub_out = p->last_n_sub;
    return HIC_OK;
}

int hic_decode_export_restarts(hic_decode_plan* p, uint8_t* h_off, uint8_t* h_cnt, uint64_t capacity, void* stream) {
    HIC_REQUIRE(p && h_off && h_cnt, "NULL argument");
    if (capacity < p->last_n_sub)
        return hic::fail(HIC_ERR_CAPACITY, "room for %llu restart records, the last run has %llu", (unsigned long long)capacity,
                         (unsigned long long)p->last_n_sub);
    if (p->last_n_sub == 0) return HIC_OK;
    cudaStream_t st = as_stream(stream);
    HIC_LAUNCH("restart_export_kernel", st, restart_export_kernel<<<(unsigned)p->last_n_tiles, SUB_PER_CTA, 0, st>>>(p->d_tiles, p->d_nbits, p->d_sub_end, p->d_sub_cnt,
                                                                  p->d_restart, p->d_restart + p->sub_capacity));
    HIC_CUDA(cudaMemcpyAsync(h_off, p->d_restart, p->last_n_sub, cudaMemcpyDeviceToHost, st));
    HIC_CUDA(cudaMemcpyAsync(h_cnt, p->d_restart + p->sub_capacity, p->last_n_sub, cudaMemcpyDeviceToHost, st));
    HIC_CUDA(cudaStreamSynchronize(st));
    return HIC_OK;
}

}  // extern "C"
